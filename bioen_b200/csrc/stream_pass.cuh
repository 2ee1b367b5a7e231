// stream_pass.cuh -- the two kernels that touch the M x N matrix yTilde.
//
// Every BioEn evaluation is two skinny products with the same fp64 matrix (SURVEY.md section 8d):
//
//   ROW pass   out_i = sum_j (y_ij [- b_i]) * v_j      "yTilde . w"       reference: c_bioen_common.c:78-83,
//                                                                          c_bioen_kernels_forces.c:330-338
//   COL pass   out_j = sum_i a_i * (y_ij [- b_i])      "yTilde^T . r"     reference: c_bioen_kernels_logw.c:197-204,
//                                                                          c_bioen_kernels_forces.c:140-147,311-318
//
// Both are HBM-bound (0.25 flop/byte) so the design goal is only: keep >100 KB of loads in flight per SM,
// read every byte of yTilde exactly once per pass, never re-read.  One persistent CTA per SM runs a
// producer/consumer ring:
//
//   * warp NW (one elected lane) is the producer: for each R x C tile it arms an mbarrier with the byte count
//     and issues one 2-D tiled TMA load (cp.async.bulk.tensor) for the matrix tile plus one or two 1-D bulk
//     copies for the slices of the small vectors the tile needs.  Tiles are 32 KB, the ring holds 4 of them
//     (128 KB in flight per SM; deeper is slower, see kStages below).  Out-of-range rows/columns are zero-filled by
//     the TMA unit, the vectors are zero-padded, so there is no tail code anywhere.
//   * warps 0..NW-1 are consumers.  Each warp owns a fixed slice of every tile (ROW: 4 rows x all columns,
//     COL: all rows x 16 columns) and keeps its fp64 accumulators in registers for a whole "run" of tiles
//     (ROW: a row-tile swept along the columns; COL: a column block swept down the rows), reads shared
//     memory with conflict-free 128-bit loads, and releases the stage with one mbarrier arrive per warp.
//     Warps never synchronise with each other.
//
// The producer / consumer roles are device functions (pass_produce / pass_consume, templates on the storage type of
// the matrix) shared by the stand-alone kernel below and by the persistent evaluation kernel (persistent_eval.cuh).
//
// Work split: tiles are numbered run-major and cut into `nCTA` equal contiguous chunks, so the load is
// balanced to +-1 tile whatever M and N are (the column pass deals whole runs round-robin instead where every CTA
// gets some: TileWalk mode 2, the default since round 2).  A run that straddles a chunk border is finished by two (or
// more) CTAs; each writes its partial sums to its own slot (`slot = cta - first_cta_of_run`), and the small
// finalize kernels (vector_kernels.cu) add the slots in a fixed order.  No atomics on data: results are
// bit-reproducible run to run.
#pragma once
#include "common.cuh"

namespace bioen {

enum PassMode { kRowPass = 0, kColPass = 1 };

constexpr int kTileR = 32;    // rows per tile
constexpr int kTileC = 128;   // columns per tile  (128 doubles = 1 KB per tile row)
// Ring depth.  MORE is not better: measured at N = 1e6 x M = 1e3 (read-only LDG stream on the same box: 7.25 TB/s)
//   2 stages 6.52, 3: 7.13, 4: 7.24, 5: 7.13, 6: 7.06 TB/s.  ~100 KB in flight per SM saturate the HBM; deeper
// queues only add contention in the memory system (the plain LDG stream shows the same: 64 KB/SM in flight 7.3 TB/s,
// 256 KB/SM 7.18 TB/s).
#ifndef BIOEN_PASS_STAGES
#define BIOEN_PASS_STAGES 4
#endif
#ifndef BIOEN_PASS_CTAS_PER_SM
#define BIOEN_PASS_CTAS_PER_SM 1
#endif
constexpr int kStages = BIOEN_PASS_STAGES;    // ring depth (fp64 storage)
constexpr int kPassCtasPerSM = BIOEN_PASS_CTAS_PER_SM;
constexpr int kConsumerWarps = 8;
constexpr int kAuxBytes = 2048;                                   // vector slices travelling with a tile
constexpr int kTileBytes = kTileR * kTileC * (int)sizeof(double);  // 32 KB
constexpr int kStageBytes = kTileBytes + kAuxBytes;
constexpr int kPassThreads = (kConsumerWarps + 1) * 32;

// Ring geometry per storage type of the matrix.  T = double is the path everything is measured and pinned on.
// T = float is the opt-in reduced-precision STORAGE of yTilde (BIOEN_B200_OPT_FP32_STORAGE): tiles are 16 KB, the
// ring is twice as deep so that the same ~128 KB per SM are in flight, every product and every sum is still fp64.
template <typename T>
struct PassGeom {
    static constexpr int kTile = kTileR * kTileC * (int)sizeof(T);
    static constexpr int kStage = kTile + kAuxBytes;
    static constexpr int kNStages = kStages * (int)(sizeof(double) / sizeof(T));
    static constexpr int kSmem = kNStages * kStage + 2 * kNStages * (int)sizeof(uint64_t) + 128;
};
constexpr int kPassSmemBytes = PassGeom<double>::kSmem;
constexpr int kPassSmemBytesF32 = PassGeom<float>::kSmem;

struct PassArgs {
    int nRT;            // number of row tiles     ceil(M / kTileR)
    int nCB;            // number of column blocks ceil(N / kTileC)
    long long T;        // nRT * nCB
    long long chunk;    // tiles per CTA (contiguous order)
    int interleave;     // column pass only, 1: whole runs are dealt round-robin to the CTAs
    int evict_first;    // 1: stream yTilde through L2 with evict_first (matrix >> L2)
    const double* vN;   // ROW: v_j, length >= nCB*kTileC, zero padded
    const double* vMb;  // ROW with SUB: b_i, length >= nRT*kTileR, zero padded
    const double* ab;   // COL: interleaved {a_i, b_i}, >= nRT*kTileR pairs, zero padded
    double* partial;    // ROW: [slot][ld] per-row partial sums; COL: [slot][ld] per-column partial sums
    long long ld;       // leading dimension of `partial`
};

// slots a run of length L starting at tile run*L occupies: first CTA and count
__host__ __device__ inline long long pass_first_cta(long long run, long long L, long long chunk) {
    return (run * L) / chunk;
}
__host__ __device__ inline int pass_num_slots(long long run, long long L, long long chunk) {
    return (int)(((run + 1) * L - 1) / chunk - (run * L) / chunk) + 1;
}

// The order in which one CTA visits its tiles.  A run is the set of tiles that accumulate into the same outputs
// (row pass: the nCB tiles of a row tile; column pass: the nRT tiles of a column block).
//   contiguous  CTA b owns tiles [b*chunk, (b+1)*chunk) of the run-major order: far-apart regions of the matrix
//               are streamed at the same time.
//   interleaved (column pass only): run r goes to CTA r mod G.  At any moment the whole chip reads one compact
//               window of the matrix (every row a contiguous stretch of ~G KB), which the DRAM serves ~2-3 % faster
//               (measured with a TMA-free read probe).  Each run has one slot, written by the CTA that owns it.
struct TileWalk {
    long long run, left, L;
    int k, G;
    bool interleaved;
    __host__ __device__ __forceinline__ void init(int pass_mode, const PassArgs& a, int b, int grid) {
        L = (pass_mode == kRowPass) ? a.nCB : a.nRT;
        G = grid;
        interleaved = a.interleave != 0;
        if (!interleaved) {
            const long long t0 = (long long)b * a.chunk;
            const long long t1 = (t0 + a.chunk < a.T) ? t0 + a.chunk : a.T;
            left = t1 > t0 ? t1 - t0 : 0;
            run = t0 / L;
            k = (int)(t0 - run * L);
        } else {
            const long long nruns = a.nCB;
            left = b < nruns ? ((nruns - b + G - 1) / G) * L : 0;
            run = b;
            k = 0;
        }
    }
    // does the current tile close the CTA's part of its run?
    __host__ __device__ __forceinline__ bool closes_run() const { return left == 1 || k + 1 == (int)L; }
    __host__ __device__ __forceinline__ void advance() {
        --left;
        if (++k == (int)L) {
            k = 0;
            run += interleaved ? G : 1;
        }
    }
    __host__ __device__ __forceinline__ long long slot(int b, long long chunk) const {
        return interleaved ? 0 : (long long)b - pass_first_cta(run, L, chunk);
    }
};

// Ring position of one role (producer or consumer) of a CTA.  It survives from one pass to the next when several
// passes run inside one kernel (persistent_eval.cuh): the mbarrier phases simply continue.
struct RingPos {
    int stage;
    uint32_t phase;
};

template <typename T = double>
__device__ __forceinline__ void pass_ring_init(unsigned char* smem) {
    using Geo = PassGeom<T>;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + Geo::kNStages * Geo::kStage);
    uint64_t* empty = full + Geo::kNStages;
    if (threadIdx.x == 0) {
        for (int s = 0; s < Geo::kNStages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kConsumerWarps);
        }
        fence_barrier_init();
    }
}

// the producer role of one pass: called by ONE lane (warp kConsumerWarps, lane 0)
template <int MODE, bool SUB, typename T = double>
__device__ __forceinline__ void pass_produce(unsigned char* smem, const CUtensorMap* tmap, const PassArgs& a,
                                             TileWalk tw, RingPos& rp) {
    using Geo = PassGeom<T>;
    constexpr int kStages = Geo::kNStages, kStageBytes = Geo::kStage, kTileBytes = Geo::kTile;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
    uint64_t* empty = full + kStages;
    const uint64_t policy = a.evict_first ? l2_policy_evict_first() : l2_policy_evict_last();
    int stage = rp.stage;
    uint32_t phase = rp.phase;
    for (; tw.left > 0; tw.advance()) {
        const int rt = (MODE == kRowPass) ? (int)tw.run : tw.k;
        const int cb = (MODE == kRowPass) ? tw.k : (int)tw.run;
        unsigned char* st = smem + (size_t)stage * kStageBytes;
        mbar_wait(&empty[stage], phase);
        uint32_t bytes = kTileBytes;
        if (MODE == kRowPass) bytes += kTileC * 8 + (SUB ? kTileR * 8 : 0);
        else bytes += kTileR * 16;
        mbar_expect_tx(&full[stage], bytes);
        tma_load_2d(st, tmap, cb * kTileC, rt * kTileR, &full[stage], policy);
        if (MODE == kRowPass) {
            bulk_load_1d(st + kTileBytes, a.vN + (size_t)cb * kTileC, kTileC * 8, &full[stage]);
            if (SUB)
                bulk_load_1d(st + kTileBytes + kTileC * 8, a.vMb + (size_t)rt * kTileR, kTileR * 8, &full[stage]);
        } else {
            bulk_load_1d(st + kTileBytes, a.ab + (size_t)rt * kTileR * 2, kTileR * 16, &full[stage]);
        }
        if (++stage == kStages) { stage = 0; phase ^= 1; }
    }
    rp.stage = stage;
    rp.phase = phase;
}

// the consumer role of one pass: called by the kConsumerWarps consumer warps
// one lane's share of a tile row in the row pass -- four columns -- and the matching slice of v
// (fp64 storage: columns {2l, 2l+1} and {64+2l, 64+2l+1}, two 16-byte loads; fp32 storage: columns 4l .. 4l+3, one)
template <typename T>
struct RowFrag;
template <>
struct RowFrag<double> {
    double2 v0, v1;
    __device__ __forceinline__ void load_v(const double2* vv, int lane) { v0 = vv[lane]; v1 = vv[32 + lane]; }
    __device__ __forceinline__ double dot(const unsigned char* rowp, int lane, bool sub, double b, double s) const {
        const double2* yr = reinterpret_cast<const double2*>(rowp);
        double2 y0 = yr[lane], y1 = yr[32 + lane];
        if (sub) { y0.x -= b; y0.y -= b; y1.x -= b; y1.y -= b; }
        s = fma(y0.x, v0.x, s);
        s = fma(y0.y, v0.y, s);
        s = fma(y1.x, v1.x, s);
        s = fma(y1.y, v1.y, s);
        return s;
    }
};
template <>
struct RowFrag<float> {
    double2 v0, v1;
    __device__ __forceinline__ void load_v(const double2* vv, int lane) { v0 = vv[2 * lane]; v1 = vv[2 * lane + 1]; }
    __device__ __forceinline__ double dot(const unsigned char* rowp, int lane, bool sub, double b, double s) const {
        const float4 y = reinterpret_cast<const float4*>(rowp)[lane];
        double y0 = (double)y.x, y1 = (double)y.y, y2 = (double)y.z, y3 = (double)y.w;
        if (sub) { y0 -= b; y1 -= b; y2 -= b; y3 -= b; }
        s = fma(y0, v0.x, s);
        s = fma(y1, v0.y, s);
        s = fma(y2, v1.x, s);
        s = fma(y3, v1.y, s);
        return s;
    }
};

template <int MODE, bool SUB, typename T = double>
__device__ __forceinline__ void pass_consume(unsigned char* smem, const PassArgs& a, TileWalk tw, RingPos& rp) {
    using Geo = PassGeom<T>;
    constexpr int kStages = Geo::kNStages, kStageBytes = Geo::kStage, kTileBytes = Geo::kTile;
    constexpr int kRowBytes = kTileC * (int)sizeof(T);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
    uint64_t* empty = full + kStages;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int stage = rp.stage;
    uint32_t phase = rp.phase;

    if (MODE == kRowPass) {
        constexpr int RPW = kTileR / kConsumerWarps;  // rows per warp = 4
        double acc[RPW];
#pragma unroll
        for (int r = 0; r < RPW; ++r) acc[r] = 0.0;
        for (; tw.left > 0; tw.advance()) {
            const unsigned char* st = smem + (size_t)stage * kStageBytes;
            mbar_wait(&full[stage], phase);
            RowFrag<T> fr;
            fr.load_v(reinterpret_cast<const double2*>(st + kTileBytes), lane);
            const double* bv = reinterpret_cast<const double*>(st + kTileBytes + kTileC * 8);
#pragma unroll
            for (int r = 0; r < RPW; ++r) {
                const int row = warp * RPW + r;
                acc[r] = fr.dot(st + (size_t)row * kRowBytes, lane, SUB, SUB ? bv[row] : 0.0, acc[r]);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[stage]);
            if (++stage == kStages) { stage = 0; phase ^= 1; }
            if (tw.closes_run()) {
                double* out = a.partial + tw.slot((int)blockIdx.x, a.chunk) * a.ld + tw.run * kTileR + warp * RPW;
#pragma unroll
                for (int r = 0; r < RPW; ++r) {
                    const double s = warp_sum(acc[r]);
                    if (lane == 0) out[r] = s;
                    acc[r] = 0.0;
                }
            }
        }
    } else {
        // warp -> 16 columns; lane -> (row group of 8 rows, column pair)
        constexpr int CPW = kTileC / kConsumerWarps;  // 16 columns per warp
        static_assert(CPW == 16 && kTileR == 32, "column-pass lane mapping assumes a 32 x 128 tile");
        const int cp = lane & 7, rg = lane >> 3;
        double acc0 = 0.0, acc1 = 0.0;
        for (; tw.left > 0; tw.advance()) {
            const unsigned char* st = smem + (size_t)stage * kStageBytes;
            mbar_wait(&full[stage], phase);
            const double2* abv = reinterpret_cast<const double2*>(st + kTileBytes);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int row = rg * 8 + q;
                double2 y;
                if (sizeof(T) == 8) {
                    y = (reinterpret_cast<const double2*>(st + (size_t)row * kRowBytes) + warp * (CPW / 2))[cp];
                } else {
                    const float2 yf = (reinterpret_cast<const float2*>(st + (size_t)row * kRowBytes) + warp * (CPW / 2))[cp];
                    y = make_double2((double)yf.x, (double)yf.y);
                }
                const double2 ab = abv[row];
                if (SUB) {
                    acc0 = fma(ab.x, y.x - ab.y, acc0);
                    acc1 = fma(ab.x, y.y - ab.y, acc1);
                } else {
                    acc0 = fma(ab.x, y.x, acc0);
                    acc1 = fma(ab.x, y.y, acc1);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[stage]);
            if (++stage == kStages) { stage = 0; phase ^= 1; }
            if (tw.closes_run()) {
                // add the four row groups in a fixed order
                acc0 += __shfl_xor_sync(0xffffffffu, acc0, 8);
                acc1 += __shfl_xor_sync(0xffffffffu, acc1, 8);
                acc0 += __shfl_xor_sync(0xffffffffu, acc0, 16);
                acc1 += __shfl_xor_sync(0xffffffffu, acc1, 16);
                if (rg == 0) {
                    double2* out = reinterpret_cast<double2*>(a.partial + tw.slot((int)blockIdx.x, a.chunk) * a.ld +
                                                              tw.run * kTileC + warp * CPW);
                    out[cp] = make_double2(acc0, acc1);
                }
                acc0 = acc1 = 0.0;
            }
        }
    }
    rp.stage = stage;
    rp.phase = phase;
}

// ------------------------------------------------------------------------------------------------
// Column pass of the log-weights gradient WITH its epilogue (single GPU, interleaved run order: every run -- a column
// block swept down all row tiles -- belongs to ONE CTA, so the warp that closes a run holds the finished
// c_j = sum_i r_i (y_ij - avg_i) of its 16 columns and can form
//     grad_j = w_j theta (g_j - <g> - G_j + <G>) + w_j c_j          (c_bioen_kernels_logw.c:214-217)
// right there instead of writing c_j for a separate O(N) kernel to read back: no partial-sum round trip through HBM
// (16 MB at N = 1e6), one kernel less, and the gradient leaves the SM while the pass is still streaming -- which is
// what lets bioen_b200_eval write it straight into page-locked host memory, overlapped with the pass.
// grad.d, ||grad||^2 and max|grad| are accumulated per lane, combined per CTA in a fixed order and finished by
// k_colgrad_finish.
// ------------------------------------------------------------------------------------------------
struct ColGradArgs {
    int n;
    const double* g;
    const double* G;
    const double* w;
    const double* d;      // may be nullptr
    double* grad;         // device memory, or page-locked host memory mapped into the device's address space
    double theta;
    const double* sc;     // scalar file: <g>, <G>
    int i_gbar, i_Gbar;
    double* cta_part;     // [gridDim.x][3]
    int i_wscale;         // >= 0 (sharded run, one exchange per half): w holds e_j, w_j = e_j * sc[i_wscale] is
    double* wio;          //      formed here and written back to wio
};

template <typename T>
__global__ void __launch_bounds__(kPassThreads, kPassCtasPerSM)
    stream_colgrad_kernel(const __grid_constant__ CUtensorMap tmap, const PassArgs a, const ColGradArgs ga) {
    using Geo = PassGeom<T>;
    constexpr int kNS = Geo::kNStages, kStageB = Geo::kStage, kTileB = Geo::kTile;
    constexpr int kRowBytes = kTileC * (int)sizeof(T);
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u);
    __shared__ double s_red[3][kConsumerWarps];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    TileWalk tw;
    tw.init(kColPass, a, (int)blockIdx.x, (int)gridDim.x);   // a.interleave must be 1 (whole runs per CTA)
    pass_ring_init<T>(smem);
    __syncthreads();
    if (warp == kConsumerWarps) {
        if (lane == 0 && tw.left > 0) {
            prefetch_tensormap(&tmap);
            RingPos rp{0, 1};
            pass_produce<kColPass, true, T>(smem, &tmap, a, tw, rp);
        }
        return;
    }
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + kNS * kStageB);
    uint64_t* empty = full + kNS;
    constexpr int CPW = kTileC / kConsumerWarps;
    const int cp = lane & 7, rg = lane >> 3;
    const double gbar = ga.sc[ga.i_gbar], Gbar = ga.sc[ga.i_Gbar];
    const double wscale = ga.i_wscale >= 0 ? ga.sc[ga.i_wscale] : 1.0;
    double acc0 = 0.0, acc1 = 0.0, dg = 0.0, gn = 0.0, gi = 0.0;
    int stage = 0;
    uint32_t phase = 0;
    for (; tw.left > 0; tw.advance()) {
        const unsigned char* st = smem + (size_t)stage * kStageB;
        mbar_wait(&full[stage], phase);
        const double2* abv = reinterpret_cast<const double2*>(st + kTileB);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int row = rg * 8 + q;
            double2 y;
            if (sizeof(T) == 8) {
                y = (reinterpret_cast<const double2*>(st + (size_t)row * kRowBytes) + warp * (CPW / 2))[cp];
            } else {
                const float2 yf = (reinterpret_cast<const float2*>(st + (size_t)row * kRowBytes) + warp * (CPW / 2))[cp];
                y = make_double2((double)yf.x, (double)yf.y);
            }
            const double2 ab = abv[row];
            acc0 = fma(ab.x, y.x - ab.y, acc0);
            acc1 = fma(ab.x, y.y - ab.y, acc1);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[stage]);
        if (++stage == kNS) { stage = 0; phase ^= 1; }
        if (tw.closes_run()) {
            acc0 += __shfl_xor_sync(0xffffffffu, acc0, 8);
            acc1 += __shfl_xor_sync(0xffffffffu, acc1, 8);
            acc0 += __shfl_xor_sync(0xffffffffu, acc0, 16);
            acc1 += __shfl_xor_sync(0xffffffffu, acc1, 16);
            if (rg == 0) {
                const long long j = tw.run * kTileC + warp * CPW + 2 * cp;
                if (j < ga.n) {
                    const bool two = j + 1 < ga.n;
                    double2 gv, Gv, wv;
                    if (two) {
                        gv = *reinterpret_cast<const double2*>(ga.g + j);
                        Gv = *reinterpret_cast<const double2*>(ga.G + j);
                        wv = *reinterpret_cast<const double2*>(ga.w + j);
                    } else {   // last column of an odd N: no access past the end of caller-owned vectors
                        gv = make_double2(ga.g[j], 0.0);
                        Gv = make_double2(ga.G[j], 0.0);
                        wv = make_double2(ga.w[j], 0.0);
                    }
                    if (ga.i_wscale >= 0) {
                        wv.x *= wscale;
                        wv.y *= wscale;
                        if (two) *reinterpret_cast<double2*>(ga.wio + j) = wv;
                        else ga.wio[j] = wv.x;
                    }
                    const double g0 = wv.x * ga.theta * (gv.x - gbar - Gv.x + Gbar) + wv.x * acc0;
                    const double g1 = two ? wv.y * ga.theta * (gv.y - gbar - Gv.y + Gbar) + wv.y * acc1 : 0.0;
                    if (two) *reinterpret_cast<double2*>(ga.grad + j) = make_double2(g0, g1);
                    else ga.grad[j] = g0;
                    if (ga.d) {
                        dg = fma(g0, ga.d[j], dg);
                        if (two) dg = fma(g1, ga.d[j + 1], dg);
                    }
                    gn = fma(g0, g0, gn);
                    gn = fma(g1, g1, gn);
                    gi = fmax(gi, fmax(fabs(g0), fabs(g1)));
                }
            }
            acc0 = acc1 = 0.0;
        }
    }
    // per-CTA partial of the three scalars (consumer warps only: the producer warp has left), fixed order
    dg = warp_sum(dg);
    gn = warp_sum(gn);
    gi = warp_max(gi);
    if (lane == 0) { s_red[0][warp] = dg; s_red[1][warp] = gn; s_red[2][warp] = gi; }
    asm volatile("bar.sync 1, %0;" ::"n"(kConsumerWarps * 32) : "memory");
    if (threadIdx.x == 0) {
        double t0 = 0.0, t1 = 0.0, t2 = 0.0;
        for (int w = 0; w < kConsumerWarps; ++w) { t0 += s_red[0][w]; t1 += s_red[1][w]; t2 = fmax(t2, s_red[2][w]); }
        ga.cta_part[3 * blockIdx.x + 0] = t0;
        ga.cta_part[3 * blockIdx.x + 1] = t1;
        ga.cta_part[3 * blockIdx.x + 2] = t2;
    }
}

// sums the per-CTA partials of stream_colgrad_kernel in CTA order; the sharded variant (with the exchange of
// {grad.d, ||grad||^2, ||x||^2, max|grad|} between the ranks) is k_colgrad_finish_sharded in vector_kernels.cuh
__global__ void __launch_bounds__(256) k_colgrad_finish(int ncta, const double* cta_part, double* sc, int i_dg,
                                                        int i_gn, int i_gi) {
    __shared__ double red[3][8];
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
        sc[i_dg] = t0;
        sc[i_gn] = t1;
        sc[i_gi] = t2;
    }
}

template <int MODE, bool SUB, typename T = double>
__global__ void __launch_bounds__(kPassThreads, kPassCtasPerSM)
    stream_pass_kernel(const __grid_constant__ CUtensorMap tmap, const PassArgs a) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // 128-byte align the ring by hand (dynamic smem base is only guaranteed 16-byte aligned)
    // offset arithmetic on the extern array (not a uintptr_t round trip) keeps the shared address space known
    // to the compiler: LDS instead of generic LD.E
    unsigned char* smem = smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    TileWalk tw;   // producer and consumers walk the same tile sequence
    tw.init(MODE, a, (int)blockIdx.x, (int)gridDim.x);
    pass_ring_init<T>(smem);
    __syncthreads();
    if (warp == kConsumerWarps) {
        if (lane == 0 && tw.left > 0) {
            prefetch_tensormap(&tmap);
            RingPos rp{0, 1};  // a fresh barrier passes a wait on parity 1
            pass_produce<MODE, SUB, T>(smem, &tmap, a, tw, rp);
        }
        return;
    }
    if (tw.left == 0) return;
    RingPos rp{0, 0};
    pass_consume<MODE, SUB, T>(smem, a, tw, rp);
}

}  // namespace bioen
