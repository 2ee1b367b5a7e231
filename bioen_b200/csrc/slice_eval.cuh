// slice_eval.cuh -- one evaluation as ONE cooperative kernel whose CTAs keep their part of yTilde in SHARED MEMORY.
//
// The problems BioEn is actually run on are small: the reference's own fixtures are 808 x 10 ... 808 x 100, the ala5
// example is 28 x 50 001 (11 MB).  persistent_eval_kernel runs such an evaluation in one launch, but it still walks the
// matrix tile by tile through the TMA ring once per pass and separates the phases by 4 (log-weights) or 7 (forces)
// grid barriers of ~2.5 us each: 42 / 59 us per evaluation at the ala5 shape, of which the matrix passes are ~10 us.
//
// Here the COLUMNS are dealt to the CTAs once (CTA c owns columns [c*nc, (c+1)*nc), all M rows: up to ~210 KB of
// shared memory), the slice is read from L2 / HBM ONCE per launch (cp.async, overlapped with the vector prologue), and
// every sweep of the evaluation -- 2 for log-weights, 4 for forces -- runs out of shared memory.  The CTAs play the
// role the ranks play in the sharded path (DESIGN.md section 5): each forms e_j = exp(x_j - m_c) with its OWN maximum,
// its partial row sums A_c,i = sum_j y_ij e_j and its part of the prior sums; ONE grid barrier later every CTA combines
// the G contributions in CTA order with exp(m_c - m) -- identical values in every CTA, so no second barrier publishes
// avg / r -- and goes on to the gradient of its own columns; the CTA that arrives last (ticket) finishes the grid
// sums.  1 barrier + 1 ticket per evaluation for both methods.
//
//   log-weights   A: x = xp + stp d, m_c, e_j, S_c, prior sums, A_c,i        | barrier |
//                 B: m, S, avg, r, chi^2, f;  w_j = e_j s_c / S;  c_j = sum_i r_i (y_ij - avg_i);  grad_j   -> ticket
//   forces        A: f = xp + stp d;  x_j = sum_i f_i y_ij;  m_c, u_j = w0_j e^{x_j - m_c}, S_c, K_c, A_c,i | barrier |
//                 B: m, S, KL, avg, r, chi^2, f;  w_j, lr_j;  t_j = sum_i r_i y_ij;  E_j;
//                    g_c,i = sum_j (y_ij - avg_i) E_j                                                      -> ticket
//                 (KL = sum_j w_j lr_j is formed from K_c = sum_j (x_j - m_c) u_j over the structures with
//                  w0_j >= DBL_MIN and U_c = sum u_j over the others, i.e. with the reference's guard lr_j = 0 for
//                  w0_j < DBL_MIN but without its guard lr_j = 0 for w_j < DBL_MIN: those terms are < 1e-305,
//                  c_bioen_kernels_forces.c:246-274)
//
// Reference lines this restates: c_bioen_kernels_logw.c:29-217, 525-561; c_bioen_kernels_forces.c:93-340.
// All reductions are fixed-order (geometry-dependent only): results are bit-reproducible run to run, and the
// gradient-only launch (mode 2, the continuation of an objective-only probe) reproduces the bits of mode 1.
#pragma once
#include "persistent_eval.cuh"

namespace bioen {

constexpr int kSliceThreads = 512;   // one CTA per SM: 16 warps hide the latency of the dependent sweeps (8 do not)
constexpr int kSliceWarps = kSliceThreads / 32;
constexpr int kSliceGP = 160;    // most CTAs of a launch
constexpr int kSliceHdr = 8;     // scalars ahead of the M row sums in a CTA's table record: m_c, S_c, the prior sums
constexpr int kSliceMinCols = 8; // fewest columns per CTA

struct SliceArgs {
    int method, mode;    // method 0 log-weights / 1 forces; mode = PEvalMode
    int M, N;
    int nc;              // columns per CTA (even)
    int ncs;             // row stride of the slice in shared memory (even, = 2 mod 4: at most 2-way bank conflicts
                         // when the lanes of a warp walk down a column)
    int ms;              // stride of a CTA's record in the tables (>= kSliceHdr + M)
    int cx_log2;         // column reduce: 2^cx_log2 threads along the columns, kSliceThreads >> cx_log2 row groups
    int l_log2;          // row reduce: 2^l_log2 lanes per row
    int lt_log2;         // table rows: 2^lt_log2 lanes per row
    const double* Y;
    long long ld;
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
    double theta;
    double* sc;
    double* tab;         // [grid][ms]   phase A: {m_c, S_c, prior sums ..., A_c,i}
    double* gtab;        // [grid][ms]   forces: gradient contributions g_c,i
    double* part;        // [grid][3]                     scalars of the final grid reduction
    unsigned long long* bar;
    unsigned int* ticket;
    unsigned long long* trace;
};

__device__ __forceinline__ void cp_async16(void* dst_smem, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit_wait_all() {
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}

__device__ __forceinline__ void slice_mark(const SliceArgs& a, int& k) {
    if (a.trace && blockIdx.x == 0 && threadIdx.x == 0) a.trace[k] = global_timer_ns();
    ++k;
}

// The one grid barrier of a launch: same sense-reversing scheme as peval_grid_barrier (arrival count + generation
// word, no host state), plus a 2 s timeout so that a defect can never hang the device: returns false on timeout.
__device__ __forceinline__ bool slice_grid_barrier(unsigned long long* bar) {
    __shared__ int s_ok;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long* count = bar;
        unsigned long long* gen = bar + 16;
        int ok = 1;
        const unsigned long long my_gen = ld_acquire_gpu_u64(gen);
        __threadfence();
        if (atomicAdd(count, 1ULL) + 1 == (unsigned long long)gridDim.x) {
            *count = 0;
            __threadfence();
            asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(gen), "l"(my_gen + 1) : "memory");
        } else {
            const unsigned long long t0 = global_timer_ns();
            while (ld_acquire_gpu_u64(gen) == my_gen) {
                if (global_timer_ns() - t0 > 2000000000ull) { ok = 0; break; }
            }
        }
        __threadfence();
        s_ok = ok;
    }
    __syncthreads();
    return s_ok != 0;
}

// block-wide maximum, result in ALL threads
__device__ __forceinline__ double slice_block_max(double v, double* red) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    v = warp_max(v);
    __syncthreads();
    if (lane == 0) red[wid] = v;
    __syncthreads();
    double m = red[0];
#pragma unroll
    for (int q = 1; q < kSliceWarps; ++q) m = fmax(m, red[q]);
    return m;
}

// out_j = sum_i coef_i (y_ij - sub_i), j < nv.   Threads are laid out CX along the columns x RS = threads / CX row
// groups (tall, narrow slices keep all threads busy); the row groups are added in a fixed order through `scratch`.
template <bool SUB>
__device__ __forceinline__ void slice_col_reduce(const double* __restrict__ sl, int ncs, int M, int nv,
                                                 const double* __restrict__ coef, const double* __restrict__ sub,
                                                 double* __restrict__ out, double* scratch, int cx_log2) {
    const int tid = threadIdx.x;
    const int CX = 1 << cx_log2, RS = kSliceThreads >> cx_log2;
    const int cx = tid & (CX - 1), rg = tid >> cx_log2;
    for (int j = cx; j < nv; j += CX) {
        double acc0 = 0.0, acc1 = 0.0;
        int i = rg;
        for (; i + RS < M; i += 2 * RS) {
            const double y0 = sl[(size_t)i * ncs + j], y1 = sl[(size_t)(i + RS) * ncs + j];
            acc0 = fma(coef[i], SUB ? y0 - sub[i] : y0, acc0);
            acc1 = fma(coef[i + RS], SUB ? y1 - sub[i + RS] : y1, acc1);
        }
        if (i < M) {
            const double y0 = sl[(size_t)i * ncs + j];
            acc0 = fma(coef[i], SUB ? y0 - sub[i] : y0, acc0);
        }
        const double acc = acc0 + acc1;
        if (RS == 1) out[j] = acc;
        else scratch[rg * CX + cx] = acc;   // RS > 1 implies nc <= CX: one column per thread
    }
    if (RS > 1) {
        __syncthreads();
        if (tid < nv) {
            double s0 = 0.0, s1 = 0.0;
            int q = 0;
            for (; q + 1 < RS; q += 2) { s0 += scratch[q * CX + tid]; s1 += scratch[(q + 1) * CX + tid]; }
            out[tid] = s0 + s1;   // RS is a power of two >= 2
        }
    }
    __syncthreads();
}

// f(i, sum_j (y_ij - sub_i) v_j) for every row i < M, called by one lane.  L = 2^l_log2 lanes share a row (the host
// picks L so that one sweep of the CTA covers about all rows: L = 1, a thread per row, for tall slices; a whole warp
// per row for flat ones); fixed-order shuffle sum.
template <bool SUB, class F>
__device__ __forceinline__ void slice_row_reduce(const double* __restrict__ sl, int ncs, int M, int nv,
                                                 const double* __restrict__ v, const double* __restrict__ sub,
                                                 int l_log2, F f) {
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int L = 1 << l_log2, RPW = 32 >> l_log2;
    const int lj = lane & (L - 1), sr = lane >> l_log2;
    const int rows_per_sweep = kSliceWarps * RPW;
    for (int base = 0; base < M; base += rows_per_sweep) {
        const int i = base + wid * RPW + sr;
        double acc0 = 0.0, acc1 = 0.0;
        if (i < M) {
            const double* row = sl + (size_t)i * ncs;
            const double s = SUB ? sub[i] : 0.0;
            int j = lj;
            for (; j + L < nv; j += 2 * L) {
                acc0 = fma(SUB ? row[j] - s : row[j], v[j], acc0);
                acc1 = fma(SUB ? row[j + L] - s : row[j + L], v[j + L], acc1);
            }
            if (j < nv) acc0 = fma(SUB ? row[j] - s : row[j], v[j], acc0);
        }
        double acc = acc0 + acc1;
        for (int o = L >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lj == 0 && i < M) f(i, acc);
    }
}

// f(i, sum_c rec_c[i] * scale[c]) for every row i < M of the per-CTA records `tab` (stride ms; scale == nullptr: plain
// sums), the contributions added in CTA order.  LT = 2^lt_log2 lanes share a row (LT = 1 for tall problems: consecutive
// threads read consecutive entries of one record, the G loads of a thread are independent and pipeline).
template <bool SCALE, class F>
__device__ __forceinline__ void slice_table_rows(const double* __restrict__ tab, int ms, int M, int G,
                                                 const double* __restrict__ scale, int lt_log2, F f) {
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int L = 1 << lt_log2, RPW = 32 >> lt_log2;
    const int lc = lane & (L - 1), sr = lane >> lt_log2;
    const int rows_per_sweep = kSliceWarps * RPW;
    for (int base = 0; base < M; base += rows_per_sweep) {
        const int i = base + wid * RPW + sr;
        double acc0 = 0.0, acc1 = 0.0;
        if (i < M) {
            // 8 independent loads in flight per thread: every CTA reads the whole table right after the barrier, and
            // with two loads per dependent step this phase was pure L2 latency (19 us at 1000 x 777)
            const double* col = tab + i;
            for (int c = lc; c < G; c += 8 * L) {
                double t[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int cc = c + u * L;
                    t[u] = cc < G ? __ldcg(col + (size_t)cc * ms) : 0.0;
                }
#pragma unroll
                for (int u = 0; u < 8; u += 2) {
                    const int ca = c + u * L, cb = ca + L;
                    if (ca < G) acc0 = SCALE ? fma(t[u], scale[ca], acc0) : acc0 + t[u];
                    if (cb < G) acc1 = SCALE ? fma(t[u + 1], scale[cb], acc1) : acc1 + t[u + 1];
                }
            }
        }
        double acc = acc0 + acc1;
        for (int o = L >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lc == 0 && i < M) f(i, acc);
    }
}

__global__ void __launch_bounds__(kSliceThreads, 1) slice_eval_kernel(const SliceArgs a) {
    extern __shared__ __align__(16) unsigned char slice_smem[];
    __shared__ double red[5 * 32];
    __shared__ double scratch[kSliceThreads];
    __shared__ double s_scale[kSliceGP];
    __shared__ double s_val[16];
    __shared__ bool s_last;
    const int tid = threadIdx.x, b = blockIdx.x, G = gridDim.x;
    const int M = a.M, nc = a.nc, ncs = a.ncs, ms = a.ms;
    const int Mp = (M + 1) & ~1;
    const int c0 = b * nc;
    const int nv = min(nc, a.N - c0);   // >= 1: the host launches ceil(N / nc) CTAs
    double* sl = reinterpret_cast<double*>(slice_smem);   // [M][ncs]
    double* vx = sl + (size_t)M * ncs;                    // [nc]  x_j (logw: g_j; forces: x_j, later lr_j)
    double* ve = vx + nc;                                 // [nc]  e_j / u_j, then w_j, then E_j (forces)
    double* vc = ve + nc;                                 // [nc]  column sums
    double* vr = vc + nc;                                 // [Mp]  coefficients of the column reduce: f_i, later r_i
    double* vavg = vr + Mp;                               // [Mp]  avg_i
    double* vobs = vavg + Mp;                             // [Mp]  Yobs_i
    double* vg = vobs + Mp;                               // [nc]  G_j (logw) / w0_j (forces)
    double* vd = vg + nc;                                 // [nc]  logw: direction d_j of the slope grad . d
    double* mytab = a.tab + (size_t)b * ms;
    int mk = 0;
    slice_mark(a, mk);

    // ---- the slice: M rows x ceil2(nv) columns, 16-byte cp.async (row starts are 16-byte aligned: ld, c0, ncs even)
    {
        const int hw = (nv + 1) >> 1;
        const double* src = a.Y + c0;
        const int total = M * hw;
        for (int idx = tid; idx < total; idx += kSliceThreads) {
            const int i = idx / hw, q = idx - i * hw;
            cp_async16(sl + (size_t)i * ncs + 2 * q, src + (size_t)i * a.ld + 2 * q);
        }
    }
    const double theta = a.theta;
    if (a.mode != kPEvalGradient)
        for (int i = tid; i < M; i += kSliceThreads) vobs[i] = a.Yobs[i];

    if (a.method == 0) {
        // =========================================================================== log-weights
        double gbar, Gbar;
        const double logS0 = (tid == 0 && b == 0) ? a.sc[SC_LOGS0] : 0.0;   // constant of the problem: fetched early
        if (a.mode != kPEvalGradient) {
            // ---- A: trial point, CTA-local maximum, e_j, S_c and the prior sums, ||x||^2
            double m = -DBL_MAX, xn = 0.0;
            for (int jj = tid; jj < nv; jj += kSliceThreads) {
                const int j = c0 + jj;
                double x;
                if (a.xp) { x = fma(a.stp, a.d[j], a.xp[j]); a.x[j] = x; }
                else x = a.x[j];
                vx[jj] = x;
                vg[jj] = a.Gv[j];
                vd[jj] = a.ddir ? a.ddir[j] : 0.0;
                xn = fma(x, x, xn);
                m = fmax(m, x);
            }
            const double mloc = slice_block_max(m, red);
            double v[5] = {0.0, 0.0, 0.0, 0.0, xn};
            for (int jj = tid; jj < nv; jj += kSliceThreads) {
                const double g = vx[jj], Gj = vg[jj];
                const double e = exp(g - mloc);
                ve[jj] = e;
                v[0] += e;
                v[1] = fma(g - Gj, e, v[1]);
                v[2] = fma(g, e, v[2]);
                v[3] = fma(Gj, e, v[3]);
            }
            block_sum<5>(v, red);
            if (tid == 0) {
                mytab[0] = mloc; mytab[1] = v[0]; mytab[2] = v[1]; mytab[3] = v[2]; mytab[4] = v[3]; mytab[5] = v[4];
            }
            cp_async_commit_wait_all();
            __syncthreads();
            slice_mark(a, mk);
            slice_row_reduce<false>(sl, ncs, M, nv, ve, nullptr, a.l_log2,
                                    [&](int i, double sum) { mytab[kSliceHdr + i] = sum; });
            slice_mark(a, mk);
            const bool ok = slice_grid_barrier(a.bar);
            slice_mark(a, mk);
            // ---- B: every CTA combines the G contributions in CTA order (identical values everywhere)
            double mc = -DBL_MAX, t[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
            if (tid < G) {   // the six scalars of CTA `tid`, one L2 round trip
                const double* rec = a.tab + (size_t)tid * ms;
                mc = __ldcg(rec);
#pragma unroll
                for (int k = 0; k < 5; ++k) t[k] = __ldcg(rec + 1 + k);
            }
            const double mx = slice_block_max(mc, red);
            if (tid < G) {
                const double s = exp(mc - mx);
                s_scale[tid] = s;
                t[0] *= s; t[1] *= s; t[2] *= s; t[3] *= s;
            }
            block_sum<5>(t, red);
            if (tid == 0) {
                const double inv = 1.0 / t[0];
                s_val[0] = t[0]; s_val[1] = inv;
                s_val[2] = t[1] * inv; s_val[3] = t[2] * inv; s_val[4] = t[3] * inv; s_val[5] = t[4];
            }
            __syncthreads();   // s_scale, s_val
            const double S = s_val[0], inv = s_val[1];
            gbar = s_val[3]; Gbar = s_val[4];
            double c[1] = {0.0};
            slice_table_rows<true>(a.tab + kSliceHdr, ms, M, G, s_scale, a.lt_log2, [&](int i, double sum) {
                const double av = sum * inv;
                const double r = av - vobs[i];
                vavg[i] = av;
                vr[i] = r;
                if (b == 0) {
                    a.avg[i] = av;
                    reinterpret_cast<double2*>(a.ab)[i] = make_double2(r, av);
                }
                c[0] = fma(r, r, c[0]);
            });
            block_sum<1>(c, red);
            if (tid == 0 && b == 0) {
                const double chi2 = 0.5 * c[0];
                const double prior = (s_val[2] - (mx + log(S)) + logS0) * theta;
                a.sc[SC_LSE_MAX] = mx; a.sc[SC_LSE_SUM] = S; a.sc[SC_XNORM2] = s_val[5];
                a.sc[SC_GMAX] = mx; a.sc[SC_S] = S;
                a.sc[SC_GBAR] = gbar; a.sc[SC_CAPGBAR] = Gbar;
                a.sc[SC_CHI2] = chi2; a.sc[SC_PRIOR] = prior;
                a.sc[SC_F] = ok ? prior + chi2 : p2p_nan();
            }
            // normalised weights of the own columns
            const double wscale = s_scale[b] * inv;
            for (int jj = tid; jj < nv; jj += kSliceThreads) {
                const double w = ve[jj] * wscale;
                ve[jj] = w;
                a.w[c0 + jj] = w;
            }
            slice_mark(a, mk);
            if (a.mode == kPEvalObjective) return;
            __syncthreads();   // vr, vavg complete
        } else {
            // gradient half of the point an objective-only launch has just evaluated
            for (int jj = tid; jj < nv; jj += kSliceThreads) {
                vx[jj] = a.x[c0 + jj];
                ve[jj] = a.w[c0 + jj];
                vg[jj] = a.Gv[c0 + jj];
                vd[jj] = a.ddir ? a.ddir[c0 + jj] : 0.0;
            }
            for (int i = tid; i < M; i += kSliceThreads) {
                const double2 q = reinterpret_cast<const double2*>(a.ab)[i];
                vr[i] = q.x;
                vavg[i] = q.y;
            }
            gbar = a.sc[SC_GBAR]; Gbar = a.sc[SC_CAPGBAR];
            cp_async_commit_wait_all();
            __syncthreads();
        }
        // ---- c_j = sum_i r_i (y_ij - avg_i);  gradient of the own columns;  the last CTA finishes the sums
        slice_col_reduce<true>(sl, ncs, M, nv, vr, vavg, vc, scratch, a.cx_log2);
        double dg = 0.0, gn = 0.0, gi = 0.0;
        for (int jj = tid; jj < nv; jj += kSliceThreads) {
            const int j = c0 + jj;
            const double w = ve[jj];
            const double gr = w * theta * (vx[jj] - gbar - vg[jj] + Gbar) + w * vc[jj];
            a.grad[j] = gr;
            dg = fma(gr, vd[jj], dg);
            gn = fma(gr, gr, gn);
            gi = fmax(gi, fabs(gr));
        }
        slice_mark(a, mk);
        double v3[3] = {dg, gn, gi};
        if (!grid_sum_max_last<2>(v3, a.part, a.ticket, red)) return;
        if (tid == 0) { a.sc[SC_DG] = v3[0]; a.sc[SC_GNORM2] = v3[1]; a.sc[SC_GINF] = v3[2]; }
        slice_mark(a, mk);
        return;
    }

    // =============================================================================== forces
    if (a.mode != kPEvalGradient) {
        // ---- A: f = xp + stp d (every CTA; CTA 0 stores it), x_j, CTA-local (max, S_c, K_c), A_c,i
        {
            double c[1] = {0.0};
            for (int i = tid; i < M; i += kSliceThreads) {
                double x;
                if (a.xp) { x = fma(a.stp, a.d[i], a.xp[i]); if (b == 0) a.x[i] = x; }
                else x = a.x[i];
                vr[i] = x;
                c[0] = fma(x, x, c[0]);
            }
            for (int jj = tid; jj < nv; jj += kSliceThreads) vg[jj] = a.Gv[c0 + jj];
            block_sum<1>(c, red);
            if (tid == 0 && b == 0) a.sc[SC_XNORM2] = c[0];
        }
        cp_async_commit_wait_all();
        __syncthreads();
        slice_mark(a, mk);
        slice_col_reduce<false>(sl, ncs, M, nv, vr, nullptr, vx, scratch, a.cx_log2);
        double m = -DBL_MAX;
        for (int jj = tid; jj < nv; jj += kSliceThreads) m = fmax(m, vx[jj]);
        const double mloc = slice_block_max(m, red);
        // S_c = sum u_j, K_c = sum (x_j - m_c) u_j over the structures with w0_j >= DBL_MIN (the reference's guard
        // lr_j = 0 otherwise), U_c = sum u_j over the others: their weight counts in S, their log-ratio does not
        double v[3] = {0.0, 0.0, 0.0};
        for (int jj = tid; jj < nv; jj += kSliceThreads) {
            const double xr = vx[jj] - mloc, w0 = vg[jj];
            const double u = w0 * exp(xr);
            ve[jj] = u;
            v[0] += u;
            if (w0 >= DBL_MIN) v[1] = fma(xr, u, v[1]);
            else v[2] += u;
        }
        block_sum<3>(v, red);
        if (tid == 0) { mytab[0] = mloc; mytab[1] = v[0]; mytab[2] = v[1]; mytab[3] = v[2]; }
        __syncthreads();   // ve complete
        slice_row_reduce<false>(sl, ncs, M, nv, ve, nullptr, a.l_log2,
                                [&](int i, double sum) { mytab[kSliceHdr + i] = sum; });
        slice_mark(a, mk);
        const bool ok = slice_grid_barrier(a.bar);
        slice_mark(a, mk);
        // ---- B: global (max, S), KL, avg, r, chi^2, objective -- in every CTA, CTA order
        double mc = -DBL_MAX, Sc = 0.0, Kc = 0.0, Uc = 0.0;
        if (tid < G) {
            const double* rec = a.tab + (size_t)tid * ms;
            mc = __ldcg(rec); Sc = __ldcg(rec + 1); Kc = __ldcg(rec + 2); Uc = __ldcg(rec + 3);
        }
        const double mx = slice_block_max(mc, red);
        double t[3] = {0.0, 0.0, 0.0};
        if (tid < G) {
            const double s = exp(mc - mx);
            s_scale[tid] = s;
            t[0] = Sc * s;
            t[1] = s * fma(mc - mx, Sc - Uc, Kc);
            t[2] = Uc * s;
        }
        block_sum<3>(t, red);
        if (tid == 0) {
            const double inv = 1.0 / t[0], logS = log(t[0]);
            s_val[0] = t[0]; s_val[1] = inv; s_val[2] = logS;
            // KL = sum_{w0_j >= DBL_MIN} w_j (x_j - m - log S) = K / S - log S (1 - U / S); U = 0 leaves the bits of K / S - log S
            s_val[3] = t[1] * inv - logS + logS * (t[2] * inv);
        }
        __syncthreads();
        const double S = s_val[0], inv = s_val[1], logS = s_val[2];
        double c[1] = {0.0};
        slice_table_rows<true>(a.tab + kSliceHdr, ms, M, G, s_scale, a.lt_log2, [&](int i, double sum) {
            const double av = sum * inv;
            const double r = av - vobs[i];
            vavg[i] = av;
            vr[i] = r;
            if (b == 0) {
                a.avg[i] = av;
                reinterpret_cast<double2*>(a.ab)[i] = make_double2(r, 0.0);
            }
            c[0] = fma(r, r, c[0]);
        });
        block_sum<1>(c, red);
        if (tid == 0 && b == 0) {
            const double chi2 = 0.5 * c[0], kl = s_val[3];
            a.sc[SC_LSE_MAX] = mx; a.sc[SC_LSE_SUM] = S; a.sc[SC_GMAX] = mx; a.sc[SC_S] = S;
            a.sc[SC_KL] = kl; a.sc[SC_CHI2] = chi2; a.sc[SC_PRIOR] = kl * theta;
            a.sc[SC_F] = ok ? kl * theta + chi2 : p2p_nan();
        }
        // w_j, guarded log-ratio (c_bioen_kernels_forces.c:156-171)
        const double wscale = s_scale[b] * inv;
        for (int jj = tid; jj < nv; jj += kSliceThreads) {
            const int j = c0 + jj;
            const double x = vx[jj], w0 = vg[jj];
            const double w = ve[jj] * wscale;
            const double lr = (w >= DBL_MIN && w0 >= DBL_MIN) ? (x - mx - logS) : 0.0;
            ve[jj] = w;
            vx[jj] = lr;
            a.w[j] = w;
            a.aux_n2[j] = lr;
            a.aux_n[j] = x;
        }
        slice_mark(a, mk);
        if (a.mode == kPEvalObjective) return;
        __syncthreads();   // vr, vavg, ve, vx complete
    } else {
        for (int jj = tid; jj < nv; jj += kSliceThreads) {
            ve[jj] = a.w[c0 + jj];
            vx[jj] = a.aux_n2[c0 + jj];
        }
        for (int i = tid; i < M; i += kSliceThreads) {
            vr[i] = reinterpret_cast<const double2*>(a.ab)[i].x;
            vavg[i] = a.avg[i];
        }
        cp_async_commit_wait_all();
        __syncthreads();
    }
    // ---- t_j = sum_i r_i y_ij;  E_j = (theta (1 + lr_j) + t_j) w_j;  g_c,i = sum_j (y_ij - avg_i) E_j
    slice_col_reduce<false>(sl, ncs, M, nv, vr, nullptr, vc, scratch, a.cx_log2);
    for (int jj = tid; jj < nv; jj += kSliceThreads) {
        const double E = ((1.0 + vx[jj]) * theta + vc[jj]) * ve[jj];
        ve[jj] = E;
        a.aux_n[c0 + jj] = E;
    }
    __syncthreads();
    {
        double* myg = a.gtab + (size_t)b * ms;
        slice_row_reduce<true>(sl, ncs, M, nv, ve, vavg, a.l_log2, [&](int i, double sum) { myg[i] = sum; });
    }
    slice_mark(a, mk);
    // the CTA that arrives last adds the contributions in CTA order
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        s_last = (atomicAdd(a.ticket, 1u) == (unsigned int)G - 1);
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    {
        double dg = 0.0, gn = 0.0, gi = 0.0;
        slice_table_rows<false>(a.gtab, ms, M, G, nullptr, a.lt_log2, [&](int i, double sum) {
            a.grad[i] = sum;
            if (a.ddir) dg = fma(sum, a.ddir[i], dg);
            gn = fma(sum, sum, gn);
            gi = fmax(gi, fabs(sum));
        });
        dg = warp_sum(dg); gn = warp_sum(gn); gi = warp_max(gi);
        const int lane = tid & 31, wid = tid >> 5;
        __syncthreads();
        if (lane == 0) { red[wid] = dg; red[32 + wid] = gn; red[64 + wid] = gi; }
        __syncthreads();
        if (wid == 0) {
            dg = warp_sum(lane < kSliceWarps ? red[lane] : 0.0);
            gn = warp_sum(lane < kSliceWarps ? red[32 + lane] : 0.0);
            gi = warp_max(lane < kSliceWarps ? red[64 + lane] : 0.0);
            if (lane == 0) {
                *a.ticket = 0;
                a.sc[SC_DG] = dg; a.sc[SC_GNORM2] = gn; a.sc[SC_GINF] = gi;
            }
        }
    }
    slice_mark(a, mk);
}

// ---- host side: geometry of a launch -------------------------------------------------------------------------
struct SlicePlan {
    bool ok = false;
    int nc = 0, ncs = 0, ms = 0, grid = 0, cx_log2 = 0, l_log2 = 0, lt_log2 = 0;
    size_t smem = 0;
};

// Columns per CTA: at least N / SMs (one CTA per SM), at least ~sqrt(N) / 2 -- after the barrier every CTA reads
// grid x M table entries, the sweeps touch M x nc slice entries, so narrow problems use fewer, wider CTAs -- and at
// least kSliceMinCols.  Not eligible when the slice does not fit in shared memory or the table gets large.
inline SlicePlan slice_plan(int M, int N, int num_sms, size_t max_dyn_smem) {
    SlicePlan p;
    auto even_up = [](long long v) { return (int)((v + 1) & ~1LL); };
    auto pow2_floor_log2 = [](long long v) { int c = 0; while ((2LL << c) <= v) ++c; return c; };
    const int sms = num_sms < kSliceGP ? num_sms : kSliceGP;
    int nc = even_up((N + sms - 1) / sms);
    int root = 1;
    while ((long long)root * root < N) ++root;
    nc = std::max(nc, even_up((root + 1) / 2));
    nc = std::max(nc, kSliceMinCols);
    const int ncs = (nc % 4 == 0) ? nc + 2 : nc;
    const int grid = (N + nc - 1) / nc;
    const size_t Mp = ((size_t)M + 1) & ~(size_t)1;
    const size_t smem = ((size_t)M * ncs + 5 * (size_t)nc + 3 * Mp) * sizeof(double);
    const int ms = (int)((kSliceHdr + (size_t)M + 15) & ~(size_t)15);
    if (smem > max_dyn_smem || grid > sms) return p;
    if ((size_t)grid * (size_t)ms * sizeof(double) > ((size_t)1 << 20)) return p;
    p.ok = true;
    p.nc = nc;
    p.ncs = ncs;
    p.ms = ms;
    p.grid = grid;
    p.smem = smem;
    int c = 0;
    while ((1 << c) < nc && (1 << c) < kSliceThreads) ++c;
    p.cx_log2 = c;                                  // min(threads, pow2ceil(nc)) threads along the columns
    const int per_row = pow2_floor_log2(std::max(1, kSliceThreads / M));   // lanes per row so that one sweep covers M
    p.l_log2 = std::min(std::min(per_row, 5), c);   // ... at most a warp, at most pow2ceil(nc)
    int g = 0;
    while ((1 << g) < grid) ++g;
    p.lt_log2 = std::min(std::min(per_row, 5), g);
    return p;
}

}  // namespace bioen
