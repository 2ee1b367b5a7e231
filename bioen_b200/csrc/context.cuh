// context.cuh -- device-resident BioEn problem: yTilde in HBM + everything one evaluation needs.
//
// HBM layout (all fp64):
//   Y        M x ld   row-major copy of yTilde, ld = N rounded up to 16 (rows start 128-byte aligned);
//                     described to the TMA unit by one 2-D tensor map {N, M} with 32 x 128 boxes
//   N-vectors         w (or E) padded with zeros to a multiple of 128 (1-D bulk copies never run off the end)
//   M-vectors         Yobs, avg, msum (+3 tail scalars), ab = interleaved {a_i, b_i}; padded to 32
//   partialA/B        [slots][Mpad] / [slots][Npad] partial sums of the two passes (slots <= 2 for the column
//                     pass on any N >= 19 k, a handful for the row pass)
//   sc[64]            the device scalar file (vector_kernels.cuh)
//
// One evaluation = 2 passes over Y (logw) or 4 (forces, unfused) + a few O(N)/O(M) kernels, all enqueued
// on one stream with no host synchronisation; the caller fetches sc[] when it needs numbers.
#pragma once
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "comm.cuh"
#include "fused_pass.cuh"
#include <atomic>
#include "persistent_eval.cuh"
#include "slice_eval.cuh"
#include "stream_pass.cuh"
#include "vector_kernels.cuh"

namespace bioen {

template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }
    void alloc(size_t count) {
        release();
        n = count;
        if (count) {
            CUDA_CHECK(cudaMalloc(&p, count * sizeof(T)));
            // cudaMemset on device memory is asynchronous and runs on the legacy default stream, which does NOT
            // order against our cudaStreamNonBlocking streams: without the wait below a kernel (or copy) that
            // writes the fresh buffer can be overtaken by the zero fill (seen as rare, unreproducible test failures)
            CUDA_CHECK(cudaMemsetAsync(p, 0, count * sizeof(T), cudaStreamLegacy));
            CUDA_CHECK(cudaStreamSynchronize(cudaStreamLegacy));
        }
    }
    // keep the allocation when the size is unchanged (contents are left as they are: callers that rely on zero
    // padding only ever write the unpadded part)
    void ensure(size_t count) {
        if (count != n || !p) alloc(count);
    }
    // at least `count` elements (never shrinks)
    void reserve(size_t count) {
        if (count > n || !p) alloc(count);
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
    }
};

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline PFN_encodeTiled get_encode_tiled() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        CUDA_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
        if (!p || q != cudaDriverEntryPointSuccess)
            throw CudaError("bioen_b200: driver does not provide cuTensorMapEncodeTiled");
        fn = reinterpret_cast<PFN_encodeTiled>(p);
    }
    return fn;
}

inline int round_up(long long a, long long b) { return (int)(((a + b - 1) / b) * b); }

// The context's settings of bioen_b200_set_option, at their defaults.  A context taken from the reuse cache gets a
// fresh record (Context::reset_for_reuse), so no setting outlives the problem it was made for.
struct ContextOptions {
    bool allow_fused = true;         // BIOEN_B200_OPT_FUSED_FORCES: 0 forces the four-pass tile kernels
    bool lazy_gradient = true;       // BIOEN_B200_OPT_LAZY_GRADIENT: minimisers may use the split (results identical)
    bool fuse_allowed = true;        // BIOEN_B200_OPT_FUSED_EXCHANGE
    int persistent_mode = -1;        // BIOEN_B200_OPT_PERSISTENT: -1 auto (by size), 0 off, 1 on
    bool lbfgs_gram_opt = false;     // BIOEN_B200_OPT_LBFGS_GRAM: coefficient-space update
    int slice_mode = -1;             // BIOEN_B200_OPT_SLICE: -1 / 1 on when the problem is eligible, 0 off
    bool lbfgs_small_opt = true;     // BIOEN_B200_OPT_LBFGS_SMALL: single-kernel update for n <= 1024
    bool lbfgs_speculative = true;   // BIOEN_B200_OPT_LBFGS_SPECULATIVE: 0 fetches the initial slope first
    bool fetch_zero_copy = true;     // BIOEN_B200_OPT_FETCH_ZEROCOPY: 0 fetches the scalar file with a copy
};

class Context {
   public:
    int M, N;            // local matrix shape (N = this rank's columns)
    long long N_total;   // all columns over all ranks
    long long ld = 0;    // row stride of Y in doubles
    int Mpad, Npad, nRT, nCB;
    bool interleave_col = false;
    // `chunk` as the readers of the column-pass partials need it (pass_num_slots)
    long long col_chunk() const { return interleave_col ? (long long)nRT : chunk; }
    int device, num_sms;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    Comm* comm = nullptr;  // not owned
    int nranks = 1;

    // pass geometry (shared by both passes)
    long long T, chunk;
    int grid, slotsA, slotsB;
    int evict_first;
    int vec_blocks_n, vec_blocks_m;

    double* Y = nullptr;
    DevBuf<double> Yown;
    CUtensorMap tmap;
    // opt-in fp32 STORAGE of the matrix (BIOEN_B200_OPT_FP32_STORAGE): the fp64 copy is released, the tile kernels
    // read 4-byte entries (half the roofline bytes) and keep every product and sum in fp64
    DevBuf<float> Y32;
    long long ld32 = 0;
    bool storage_fp32 = false;
    bool has_matrix() const { return Y != nullptr || storage_fp32; }
    double matrix_bytes() const { return storage_fp32 ? (double)M * ld32 * 4.0 : (double)M * (double)ld * 8.0; }

    DevBuf<double> partialA, partialB, ab, avg, msum, Yobs, w, aux_n, aux_n2, Gv, sc, red_partials, lse_all;
    DevBuf<unsigned int> ticket;
    // persistent cooperative evaluation kernel (persistent_eval.cuh)
    DevBuf<double> pe_part;
    DevBuf<unsigned long long> pe_bar;
    bool coop_ok = false;
    static constexpr double kPersistentMaxBytes = 0.6e9;   // auto: matrices up to this size per GPU
    long long persistent_launches = 0;
    DevBuf<double> colgrad_part;           // per-CTA scalars of the column pass with the gradient epilogue
    // shared-memory-resident evaluation kernel for small matrices (slice_eval.cuh)
    DevBuf<double> slice_tab, slice_gtab, slice_part;
    SlicePlan slice_pl;
    bool slice_coop = false;
    long long slice_launches = 0;
    double* h_sc = nullptr;  // pinned

    // structure-major copy + geometry of the fused two-pass forces kernels (fused_pass.cuh)
    DevBuf<double> Yt, fpart, flse;
    DevBuf<double> lbfgs_store;   // g, xp, gp, d, s[m], y[m] of the device L-BFGS (lbfgs.cuh)
    DevBuf<double> lbfgs_gram, lbfgs_gram_partials;   // coefficient-space update (BIOEN_B200_OPT_LBFGS_GRAM)
    long long ldt = 0, f_nslab = 0, f_chunk = 0;
    int f_C = 0, f_stages = 0, f_grid = 0, f_KI = 0, f_smem = 0, f_T = 1, f_rows = 0, f_rows_per_cta = 1;
    bool f_team = false;
    bool fused_ready = false, yt_valid = false;
    ContextOptions options;
    double theta = 0.0;
    bool have_logw = false, have_forces = false;
    long long passes_launched = 0, kernels_launched = 0;

    Context(int m, int n, int dev, cudaStream_t user_stream = nullptr) : M(m), N(n), N_total(n), device(dev) {
        if (m <= 0 || n <= 0) throw std::invalid_argument("bioen_b200: matrix dimensions must be positive");
        CUDA_CHECK(cudaSetDevice(device));
        cudaDeviceProp prop;
        CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
        if (prop.major < 10)
            throw CudaError("bioen_b200: this library is built for sm_100a (Blackwell B200) only");
        num_sms = prop.multiProcessorCount;
        if (user_stream) {
            stream = user_stream;
            own_stream = false;
        } else {
            CUDA_CHECK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        }
        nRT = (M + kTileR - 1) / kTileR;
        nCB = (N + kTileC - 1) / kTileC;
        Mpad = nRT * kTileR;
        Npad = nCB * kTileC;
        T = (long long)nRT * nCB;
        const long long want_cta = (long long)num_sms * kPassCtasPerSM;
        const long long ncta = T < want_cta ? T : want_cta;
        chunk = (T + ncta - 1) / ncta;
        grid = (int)((T + chunk - 1) / chunk);
        auto slots = [&](long long L) {
            long long s = (L - 1) / chunk + 2;
            return (int)(s < grid ? s : grid);
        };
        // tile order of the matrix passes (stream_pass.cuh, TileWalk).  Interleaved = the whole chip reads one compact
        // window of the matrix at a time.  Measured at N = 1e6 x M = 1e3, 40 steps each, one box, back to back
        // (round 2): contiguous 431.6 evals/s (2.3171 ms), column pass interleaved 435.4 (2.2970 ms), row pass
        // interleaved 426.7 (2.3434 ms: 148 partial-sum slots per row tile), both 430.2.  So the COLUMN pass deals its
        // runs round-robin (needs nCB >= 4 * grid), the row pass keeps contiguous chunks.
        interleave_col = nCB >= 4LL * grid;
        slotsA = slots(nCB);
        slotsB = slots(nRT);
        const int vb = 4;   // resident 256-thread blocks per SM for the O(N) kernels (measured: 2, 8, 16 are no faster)
        vec_blocks_n = std::min((N + kVecThreads - 1) / kVecThreads, num_sms * vb);
        vec_blocks_m = std::min((M + kVecThreads - 1) / kVecThreads, num_sms * vb);

        partialA.alloc((size_t)slotsA * Mpad);
        partialB.alloc((size_t)slotsB * Npad);
        ab.alloc((size_t)2 * Mpad);
        avg.alloc(Mpad);
        msum.alloc(Mpad + 16);
        Yobs.alloc(Mpad);
        w.alloc(Npad + 8);   // +8: the fused kernels copy 16-byte windows that may end one element past N
        sc.alloc(SC_COUNT);
        red_partials.alloc((size_t)std::max(vec_blocks_n, vec_blocks_m) * 4 + 16);
        ticket.alloc(4);
        lse_all.alloc(2 * 64);
        CUDA_CHECK(cudaHostAlloc(&h_sc, (SC_COUNT + 8) * sizeof(double), cudaHostAllocDefault));
        memset(h_sc, 0, (SC_COUNT + 8) * sizeof(double));   // [SC_COUNT + 1] fetch sequence number
        CUDA_CHECK(cudaFuncSetAttribute(stream_pass_kernel<kRowPass, false>,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, kPassSmemBytes));
        CUDA_CHECK(cudaFuncSetAttribute(stream_pass_kernel<kRowPass, true>,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, kPassSmemBytes));
        CUDA_CHECK(cudaFuncSetAttribute(stream_pass_kernel<kColPass, false>,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, kPassSmemBytes));
        CUDA_CHECK(cudaFuncSetAttribute(stream_pass_kernel<kColPass, true>,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, kPassSmemBytes));
        CUDA_CHECK(cudaFuncSetAttribute(stream_pass_kernel<kRowPass, false, float>,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, kPassSmemBytesF32));
        CUDA_CHECK(cudaFuncSetAttribute(stream_pass_kernel<kRowPass, true, float>,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, kPassSmemBytesF32));
        CUDA_CHECK(cudaFuncSetAttribute(stream_pass_kernel<kColPass, false, float>,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, kPassSmemBytesF32));
        CUDA_CHECK(cudaFuncSetAttribute(stream_pass_kernel<kColPass, true, float>,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, kPassSmemBytesF32));
        CUDA_CHECK(cudaFuncSetAttribute(stream_colgrad_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        kPassSmemBytes));
        CUDA_CHECK(cudaFuncSetAttribute(stream_colgrad_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        kPassSmemBytesF32));
        colgrad_part.alloc((size_t)grid * 3 + 8);
        CUDA_CHECK(cudaFuncSetAttribute(persistent_eval_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        kPassSmemBytes));
        CUDA_CHECK(cudaFuncSetAttribute(persistent_eval_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        kPassSmemBytesF32));
        pe_part.alloc((size_t)grid * kPSlots + 16);
        pe_bar.alloc(32);   // [0] arrival counter, [16] released barrier number (separate 128-byte lines)
        {
            int coop = 0, per_sm = 0;
            CUDA_CHECK(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device));
            CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, persistent_eval_kernel<float>,
                                                                     kPEvalThreads, kPassSmemBytesF32));
            coop_ok = coop && (long long)per_sm * num_sms >= grid;
            // slice kernel: plan once per context (M, N are fixed), tables only when the problem is eligible
            cudaFuncAttributes fa{};
            int optin = 0;
            CUDA_CHECK(cudaFuncGetAttributes(&fa, slice_eval_kernel));
            CUDA_CHECK(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
            const long long max_dyn = (long long)optin - (long long)fa.sharedSizeBytes - 256;
            if (max_dyn > 0) slice_pl = slice_plan(M, N, num_sms, (size_t)max_dyn);
            if (slice_pl.ok) {
                CUDA_CHECK(cudaFuncSetAttribute(slice_eval_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                (int)max_dyn));
                int occ = 0;
                CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, slice_eval_kernel, kSliceThreads,
                                                                         slice_pl.smem));
                slice_coop = coop && (long long)occ * num_sms >= slice_pl.grid;
                slice_tab.alloc((size_t)slice_pl.grid * slice_pl.ms);
                slice_gtab.alloc((size_t)slice_pl.grid * slice_pl.ms);
                slice_part.alloc((size_t)kSliceGP * 3 + 8);
            }
        }
    }

    ~Context() {
        if (h_sc) cudaFreeHost(h_sc);
        release_upload_lanes();
        for (cudaEvent_t e : pass_ev) cudaEventDestroy(e);
        if (fetch_ev) cudaEventDestroy(fetch_ev);
        if (own_stream && stream) cudaStreamDestroy(stream);
    }

    // forget the problem but keep every allocation (stateless reference entry points reuse a cached context)
    void reset_for_reuse() {
        ++eval_gen;
        sync();
        have_logw = have_forces = false;
        fused_ready = false;
        yt_valid = false;
        options = ContextOptions{};
        eval_fused = false;
        forces_x = nullptr;
        comm = nullptr;
        nranks = 1;
        N_total = N;
        Y = nullptr;
        storage_fp32 = false;
        Y32.release();
        yt_only = false;
        passes_launched = kernels_launched = 0;
        pass_timing = false;
    }
    void set_comm(Comm* c) {
        comm = c;
        nranks = c ? c->nranks : 1;
        if (nranks > 64) throw std::invalid_argument("bioen_b200: at most 64 ranks");
    }

    // ---- matrix -------------------------------------------------------------------------------
    void upload_matrix(const double* host, size_t ld_host) {
        NvtxRange nvtx("bioen:upload_ytilde");
        ld = round_up(N, 16);
        if (Yown.n != (size_t)M * ld || !Yown.p) {
            Yown.release();
            CUDA_CHECK(cudaMalloc(&Yown.p, (size_t)M * ld * sizeof(double)));
            Yown.n = (size_t)M * ld;
        }
        Y = Yown.p;
        if (ld != N) CUDA_CHECK(cudaMemsetAsync(Y, 0, (size_t)M * ld * sizeof(double), stream));
        sync();
        const size_t total = (size_t)M * N * sizeof(double);
        cudaPointerAttributes attr{};
        const bool pinned = cudaPointerGetAttributes(&attr, host) == cudaSuccess && attr.type == cudaMemoryTypeHost;
        cudaGetLastError();
        if (pinned || total < ((size_t)256 << 20)) {
            CUDA_CHECK(cudaMemcpy2DAsync(Y, ld * sizeof(double), host, ld_host * sizeof(double),
                                         (size_t)N * sizeof(double), M, cudaMemcpyHostToDevice, stream));
            sync();
        } else {
            upload_staged(host, ld_host);
        }
        make_tensor_map();
    }
    // Large pageable source (a NumPy array): a plain cudaMemcpy is limited by the driver's single-threaded staging
    // (~10 GB/s).  Here kUpThreads host threads copy row chunks into their own pinned double buffers and push them
    // with async copies on their own streams, so the host memcpy and the PCIe transfer overlap and scale.
    // 8 threads: measured on a 16-core box (8 GB, pageable NumPy source, lanes warm): 4 threads 0.72-0.79 s, 6 0.58 s,
    // 8 0.48-0.50 s, 12 0.57-0.62 s, 16 0.64-1.05 s
    static constexpr int kUpThreads = 8;
    // page-locked staging of the upload threads: allocated on first use and kept with the context (cudaHostAlloc of
    // 12 x 32 MB costs more than copying 1 GB; a caller that streams a large host matrix through this context chunk
    // by chunk -- Problem.average_streamed -- would otherwise pay it per chunk)
    struct UploadLane {
        char* stage[2] = {nullptr, nullptr};
        cudaEvent_t done[2] = {nullptr, nullptr};
        cudaStream_t st = nullptr;
        size_t bytes = 0;
    };
    std::vector<UploadLane> up_lanes;
    void release_upload_lanes() {
        for (auto& l : up_lanes) {
            for (int b = 0; b < 2; ++b) {
                if (l.stage[b]) cudaFreeHost(l.stage[b]);
                if (l.done[b]) cudaEventDestroy(l.done[b]);
            }
            if (l.st) cudaStreamDestroy(l.st);
        }
        up_lanes.clear();
    }
    void upload_staged(const double* host, size_t ld_host) {
        const size_t row_bytes = (size_t)N * sizeof(double);
        const size_t buf_bytes = std::max(row_bytes, (size_t)32 << 20);
        const int rows_per_chunk = (int)std::max<size_t>(1, buf_bytes / row_bytes);
        const int nchunks = (M + rows_per_chunk - 1) / rows_per_chunk;
        const int nthreads = std::min(kUpThreads, nchunks);
        const size_t lane_bytes = (size_t)rows_per_chunk * row_bytes;
        if ((int)up_lanes.size() < nthreads || (!up_lanes.empty() && up_lanes[0].bytes < lane_bytes)) {
            release_upload_lanes();
            up_lanes.resize(nthreads);
            for (auto& l : up_lanes) {
                CUDA_CHECK(cudaStreamCreateWithFlags(&l.st, cudaStreamNonBlocking));
                for (int b = 0; b < 2; ++b) {
                    CUDA_CHECK(cudaHostAlloc((void**)&l.stage[b], lane_bytes, cudaHostAllocDefault));
                    CUDA_CHECK(cudaEventCreateWithFlags(&l.done[b], cudaEventDisableTiming));
                }
                l.bytes = lane_bytes;
            }
        }
        std::vector<std::thread> pool;
        std::vector<std::string> errors(nthreads);
        for (int t = 0; t < nthreads; ++t) {
            pool.emplace_back([&, t] {
                try {
                    CUDA_CHECK(cudaSetDevice(device));
                    UploadLane& l = up_lanes[t];
                    int use = 0;
                    for (int c = t; c < nchunks; c += nthreads, use ^= 1) {
                        const int r0 = c * rows_per_chunk, nr = std::min(rows_per_chunk, M - r0);
                        CUDA_CHECK(cudaEventSynchronize(l.done[use]));   // the previous copy out of this buffer
                        for (int r = 0; r < nr; ++r)
                            memcpy(l.stage[use] + (size_t)r * row_bytes, host + (size_t)(r0 + r) * ld_host, row_bytes);
                        CUDA_CHECK(cudaMemcpy2DAsync(Y + (size_t)r0 * ld, ld * sizeof(double), l.stage[use], row_bytes,
                                                     row_bytes, nr, cudaMemcpyHostToDevice, l.st));
                        CUDA_CHECK(cudaEventRecord(l.done[use], l.st));
                    }
                    CUDA_CHECK(cudaStreamSynchronize(l.st));
                } catch (const std::exception& e) {
                    errors[t] = e.what();
                }
            });
        }
        for (auto& th : pool) th.join();
        for (auto& e : errors)
            if (!e.empty()) throw CudaError(e);
    }
    // allocate an uninitialised device matrix (filled by the on-device generator)
    void alloc_matrix() {
        ld = round_up(N, 16);
        Yown.release();
        CUDA_CHECK(cudaMalloc(&Yown.p, (size_t)M * ld * sizeof(double)));
        Yown.n = (size_t)M * ld;
        Y = Yown.p;
        CUDA_CHECK(cudaMemsetAsync(Y, 0, (size_t)M * ld * sizeof(double), stream));
        make_tensor_map();
    }
    // use a matrix that already lives in HBM (row stride `ld_dev` doubles, must be even; base 16-byte aligned)
    void adopt_matrix(double* dev, size_t ld_dev) {
        if ((ld_dev & 1) || (reinterpret_cast<uintptr_t>(dev) & 15))
            throw std::invalid_argument("bioen_b200: adopted yTilde needs an even row stride and a 16-byte aligned base");
        if (ld_dev < (size_t)N) throw std::invalid_argument("bioen_b200: row stride smaller than N");
        Yown.release();
        Y = dev;
        ld = (long long)ld_dev;
        make_tensor_map();
    }
    void make_tensor_map() {
        const cuuint64_t gdim[2] = {(cuuint64_t)N, (cuuint64_t)M};
        const cuuint64_t gstride[1] = {(cuuint64_t)ld * sizeof(double)};
        const cuuint32_t box[2] = {(cuuint32_t)kTileC, (cuuint32_t)kTileR};
        const cuuint32_t estr[2] = {1, 1};
        CUresult r = get_encode_tiled()(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, Y, gdim, gstride, box, estr,
                                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            char buf[128];
            snprintf(buf, sizeof buf, "bioen_b200: cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
            throw CudaError(buf);
        }
        fused_ready = false;   // the structure-major copy (if any) belongs to the previous matrix
        yt_valid = false;
        storage_fp32 = false;  // a new fp64 matrix has arrived
        Y32.release();
        // a matrix that fits in L2 with room to spare is kept there between the two passes
        evict_first = ((double)M * (double)ld * 8.0 > 80.0e6) ? 1 : 0;
    }

    // Replace the resident fp64 matrix by an fp32 copy (irreversible for this matrix).  The fused forces kernels
    // and the theta scan read the structure-major fp64 copy and are not available afterwards: the forces method runs
    // on the four tile passes (the same bytes as two fp64 passes).
    void convert_to_fp32() {
        if (storage_fp32) return;
        require_row_major("the fp32 storage option");
        if (!Y) throw std::logic_error("bioen_b200: yTilde has not been uploaded");
        ++eval_gen;
        ld32 = round_up(N, 32);
        Y32.alloc((size_t)M * ld32);
        k_convert_f32<<<num_sms * 8, 256, 0, stream>>>(Y, ld, M, N, Y32.p, ld32);
        CUDA_CHECK(cudaGetLastError());
        ++kernels_launched;
        sync();
        Yown.release();           // an adopted matrix stays with its owner
        Y = nullptr;
        Yt.release();
        fused_ready = false;
        yt_valid = false;
        storage_fp32 = true;
        const cuuint64_t gdim[2] = {(cuuint64_t)N, (cuuint64_t)M};
        const cuuint64_t gstride[1] = {(cuuint64_t)ld32 * sizeof(float)};
        const cuuint32_t box[2] = {(cuuint32_t)kTileC, (cuuint32_t)kTileR};
        const cuuint32_t estr[2] = {1, 1};
        CUresult r = get_encode_tiled()(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, Y32.p, gdim, gstride, box, estr,
                                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) throw CudaError("bioen_b200: cuTensorMapEncodeTiled (fp32) failed");
        evict_first = (matrix_bytes() > 80.0e6) ? 1 : 0;
    }

    // ---- per-method constant data ------------------------------------------------------------------
    void h2d(double* dst, const double* src, size_t n) {
        CUDA_CHECK(cudaMemcpyAsync(dst, src, n * sizeof(double), cudaMemcpyHostToDevice, stream));
    }
    void d2h(double* dst, const double* src, size_t n) {
        CUDA_CHECK(cudaMemcpyAsync(dst, src, n * sizeof(double), cudaMemcpyDeviceToHost, stream));
    }
    void d2d(double* dst, const double* src, size_t n) {
        CUDA_CHECK(cudaMemcpyAsync(dst, src, n * sizeof(double), cudaMemcpyDeviceToDevice, stream));
    }
    void sync() { CUDA_CHECK(cudaStreamSynchronize(stream)); }

    void set_observations(const double* Y_host) { h2d(Yobs.p, Y_host, M); }
    void set_theta(double th) { theta = th; ++eval_gen; }

    // logw: reference log-weights G (this rank's slice); log s0 = log sum_j exp(G_j) over ALL ranks
    void set_logw(const double* G_host, bool on_device = false) {
        require_row_major("the log-weights method");
        ++eval_gen;
        Gv.ensure(Npad + 8);
        if (on_device) d2d(Gv.p, G_host, N); else h2d(Gv.p, G_host, N);
        aux_n.ensure(Npad + 8);  // scratch x for the lse of G
        d2d(aux_n.p, Gv.p, N);
        launch_lse(aux_n.p, nullptr, nullptr, 0.0, nullptr, false);
        gather_lse();
        // log s0 = M + log S from the (gathered) pairs; tiny host round trip, once per problem
        std::vector<double> pairs(2 * nranks);
        d2h(pairs.data(), lse_pairs(), 2 * nranks);
        sync();
        double Mx = pairs[0], S = pairs[1];
        for (int r = 1; r < nranks; ++r) {
            const double mm = std::max(Mx, pairs[2 * r]);
            S = S * std::exp(Mx - mm) + pairs[2 * r + 1] * std::exp(pairs[2 * r] - mm);
            Mx = mm;
        }
        const double logs0 = Mx + std::log(S);
        CUDA_CHECK(cudaMemcpyAsync(sc.p + SC_LOGS0, &logs0, sizeof(double), cudaMemcpyHostToDevice, stream));
        sync();
        have_logw = true;
        have_forces = false;   // Gv (G vs w0) and the aux vectors are shared by the two methods
    }
    // forces: reference weights w0 (this rank's slice)
    void set_forces(const double* w0_host, bool on_device = false) {
        ++eval_gen;
        Gv.ensure(Npad + 8);      // holds w0
        if (on_device) d2d(Gv.p, w0_host, N); else h2d(Gv.p, w0_host, N);
        aux_n.ensure(Npad + 8);   // x_j, later E_j (zero padded: it feeds the row pass)
        aux_n2.ensure(Npad + 8);  // lr_j
        have_forces = true;
        have_logw = false;        // Gv now holds w0
        if (options.allow_fused && (Y || yt_only) && !storage_fp32 && !fused_ready) prepare_fused();
        if (yt_only && !fused_ready)
            throw std::logic_error("bioen_b200: structure-major-only mode: the fused forces kernels are not available "
                                   "for this problem (BIOEN_B200_OPT_FUSED_FORCES = 0, or M outside 256..~5500)");
    }

    // ---- fused two-pass forces path ------------------------------------------------------------------------
    bool fused_eligible() const {
        const long long l = (M + 1LL) & ~1LL;
        return !storage_fp32 && M >= kFMinM && l <= kFMaxLdt;
    }
    // ---- structure-major ONLY (BIOEN_B200_OPT_STRUCTURE_MAJOR_ONLY) ----------------------------------------------
    // The forces method on the fused two-pass kernels reads nothing but Yt.  In this mode the context never holds
    // the row-major matrix: uploads are transposed chunk by chunk through a small staging buffer, the generator
    // writes Yt directly, an existing matrix is transposed once and released.  Half the HBM of the default forces
    // set-up (both layouts): N = 1e6 x M = 1e3 needs 8 GB instead of 16, config 5 (400 GB) fits 4 GPUs.  Available:
    // forces evaluations and minimisers, weights, averages (through the fused kernels), downloads.  Everything that
    // streams the row-major matrix (log-weights method, tile / persistent / slice kernels, theta scan, row-affine
    // transforms, given-weights entry points) raises.
    bool yt_only = false;
    DevBuf<double> yt_stage;
    void require_row_major(const char* what) const {
        if (yt_only)
            throw std::logic_error(std::string("bioen_b200: ") + what + " needs the row-major matrix, which this context "
                                   "does not hold (BIOEN_B200_OPT_STRUCTURE_MAJOR_ONLY: forces method on the fused kernels only)");
    }
    void alloc_yt() {
        ldt = (M + 1LL) & ~1LL;
        if (Yt.n != (size_t)N * ldt || !Yt.p) {
            Yt.release();
            CUDA_CHECK(cudaMalloc(&Yt.p, (size_t)N * ldt * sizeof(double)));
            Yt.n = (size_t)N * ldt;
        }
        CUDA_CHECK(cudaMemsetAsync(Yt.p, 0, (size_t)N * ldt * sizeof(double), stream));   // pad column (odd M) stays 0
        yt_valid = true;
        fused_ready = false;
        evict_first = ((double)N * (double)ldt * 8.0 > 80.0e6) ? 1 : 0;
    }
    void enter_yt_only() {
        if (yt_only) return;
        if (storage_fp32) throw std::logic_error("bioen_b200: structure-major-only mode needs the fp64 matrix");
        if (!fused_eligible())
            throw std::invalid_argument("bioen_b200: structure-major-only mode needs the fused forces kernels "
                                        "(256 <= M <= 8192)");
        ++eval_gen;
        if (Y) {   // a row-major matrix is resident: one transposition, then it goes (an adopted one stays with its owner)
            if (!yt_valid) make_transposed();
            sync();
            Y = nullptr;
            fused_ready = false;
        }
        Yown.release();   // also the allocation a reused (cached) context kept from its previous problem
        yt_only = true;
        have_logw = false;
    }
    // rows [row0, row0 + nrows) of the HOST matrix -> Yt, staged through <= 256 MB of device memory
    void upload_rows_yt(int row0, int nrows, const double* host, size_t ld_host) {
        if (!Yt.p || !yt_valid) alloc_yt();
        const long long lds = round_up(N, 2);
        const int rows_per_chunk = (int)std::max<long long>(1, std::min<long long>(nrows, ((long long)256 << 20) / (lds * 8)));
        yt_stage.reserve((size_t)rows_per_chunk * lds);
        for (int r = 0; r < nrows; r += rows_per_chunk) {
            const int nr = std::min(rows_per_chunk, nrows - r);
            CUDA_CHECK(cudaMemcpy2DAsync(yt_stage.p, lds * sizeof(double), host + (size_t)r * ld_host,
                                         ld_host * sizeof(double), (size_t)N * sizeof(double), nr,
                                         cudaMemcpyHostToDevice, stream));
            dim3 g((unsigned)((N + 31) / 32), (unsigned)((nr + 31) / 32));
            k_transpose_block<<<g, 256, 0, stream>>>(yt_stage.p, lds, nr, N, Yt.p, ldt, row0 + r);
            CUDA_CHECK(cudaGetLastError());
            ++kernels_launched;
            sync();   // the staging buffer is reused by the next chunk (and the host rows may be pageable)
        }
        ++eval_gen;
    }
    // block [row0, row0+nrows) x [col0, col0+ncols) of Yt -> host, row-major
    void download_yt(int row0, int nrows, long long col0, long long ncols, double* out_host) {
        if (!Yt.p || !yt_valid) throw std::logic_error("bioen_b200: no matrix");
        const int rows_per_chunk = (int)std::max<long long>(1, std::min<long long>(nrows, ((long long)256 << 20) / (ncols * 8)));
        yt_stage.reserve((size_t)rows_per_chunk * ncols);
        for (int r = 0; r < nrows; r += rows_per_chunk) {
            const int nr = std::min(rows_per_chunk, nrows - r);
            dim3 g((unsigned)((ncols + 31) / 32), (unsigned)((nr + 31) / 32));
            k_gather_block<<<g, 256, 0, stream>>>(Yt.p, ldt, row0 + r, nr, col0, ncols, yt_stage.p, ncols);
            CUDA_CHECK(cudaGetLastError());
            CUDA_CHECK(cudaMemcpyAsync(out_host + (size_t)r * ncols, yt_stage.p, (size_t)nr * ncols * sizeof(double),
                                       cudaMemcpyDeviceToHost, stream));
            sync();
        }
    }

    // structure-major copy Yt[j][i] of the resident matrix (the reference's yTildeT cache, made on the device)
    void make_transposed() {
        NvtxRange nvtx("bioen:transpose_ytilde");
        if (storage_fp32)
            throw std::logic_error("bioen_b200: the structure-major copy (fused forces kernels, theta scan) needs the "
                                   "fp64 matrix; it was released by BIOEN_B200_OPT_FP32_STORAGE");
        if (!Y) throw std::logic_error("bioen_b200: yTilde has not been uploaded");
        ldt = (M + 1LL) & ~1LL;
        if (Yt.n != (size_t)N * ldt || !Yt.p) {
            Yt.release();
            CUDA_CHECK(cudaMalloc(&Yt.p, (size_t)N * ldt * sizeof(double)));
            Yt.n = (size_t)N * ldt;
        }
        yt_valid = true;
        dim3 grid((unsigned)((N + 31) / 32), (unsigned)((ldt + 31) / 32));
        k_transpose<<<grid, 256, 0, stream>>>(Y, ld, M, N, Yt.p, ldt);
        CUDA_CHECK(cudaGetLastError());
        ++kernels_launched;
    }
    void prepare_fused() {
        if (!fused_eligible()) return;
        ldt = (M + 1LL) & ~1LL;
        const long long row_bytes = ldt * 8;
        const long long smem_max = 232448 - 128;   // 227 KB opt-in limit minus our alignment slack
        f_team = false;
        if (ldt <= kTMaxLdt) {
            // team variant: T warps per structure, 8/T independent teams per CTA.  Measured at M = 1000:
            // T = 1 (eight independent warps) 1.28 ms per pass, T = 2 1.34 ms, T = 4 2.1 ms.
            f_T = ldt <= 1024 ? 1 : ldt <= 2048 ? 2 : ldt <= 4096 ? 4 : 8;
            const int teams = kTWarps / f_T;
            const long long need = (ldt + 64LL * f_T - 1) / (64LL * f_T);
            f_KI = need <= 4 ? 4 : need <= 8 ? 8 : 16;
            f_C = (int)std::max(1LL, std::min((long long)kFCMax, 8192LL / row_bytes));
            const long long stage_bytes = (((long long)f_C * row_bytes + 127) & ~127LL) + kTAuxBytes;
            const long long fixed = 2 * row_bytes + 2 * kTMaxRing * 8 + 2LL * kTWarps * 8 + 256;
            long long st = std::min((long long)kTMaxRing / teams, (smem_max - fixed) / (teams * stage_bytes));
            // ring depth: enough slabs in flight to cover the HBM latency, not more -- about 128 KB of ring per SM
            // (measured at M = 1000: 2 stages per team = 130 KB ring 6.86 TB/s, 3 stages = 195 KB 6.56 TB/s; the
            // tile kernels show the same optimum, see stream_pass.cuh)
            {
                const long long per_stage = teams * stage_bytes;
                const long long want = std::max(2LL, (131072 + per_stage / 2) / per_stage);
                st = std::min(st, want);
            }
            if (st >= 2) {
                f_team = true;
                f_stages = (int)st;
                f_rows_per_cta = 1;   // the kernel combines its teams before writing
                f_smem = (int)(teams * st * stage_bytes + fixed) + 128;
            }
        }
        if (!f_team) return;   // does not fit shared memory (M > ~5500): the four-pass tile kernels are used
        if (!yt_valid) make_transposed();
        f_nslab = ((long long)N + f_C - 1) / f_C;
        f_grid = (int)std::min<long long>(num_sms, f_nslab);
        f_chunk = (f_nslab + f_grid - 1) / f_grid;
        f_grid = (int)((f_nslab + f_chunk - 1) / f_chunk);
        f_rows = f_grid * f_rows_per_cta;
        fpart.ensure((size_t)f_rows * Mpad);
        flse.ensure((size_t)2 * f_rows);
        set_fused_attr();
        fused_ready = true;
    }
    template <int KI, int T>
    void set_team_attr() {
        CUDA_CHECK(cudaFuncSetAttribute(fused_team_pass<KI, T, kFusedSoftmaxAvg>,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, f_smem));
        CUDA_CHECK(cudaFuncSetAttribute(fused_team_pass<KI, T, kFusedGradient>,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, f_smem));
        // also loads the two kernels now (lazy module loading must not happen inside a collective operation of an
        // in-process group, see preload_kernels in bioen_b200.cu)
        cudaFuncAttributes at;
        CUDA_CHECK(cudaFuncGetAttributes(&at, fused_team_pass<KI, T, kFusedSoftmaxAvg>));
        CUDA_CHECK(cudaFuncGetAttributes(&at, fused_team_pass<KI, T, kFusedGradient>));
    }
#define BIOEN_TEAM_DISPATCH(FN)                                   \
    do {                                                          \
        if (f_T == 1 && f_KI == 4) { FN(4, 1); }                  \
        else if (f_T == 1 && f_KI == 8) { FN(8, 1); }             \
        else if (f_T == 1) { FN(16, 1); }                         \
        else if (f_T == 2 && f_KI == 4) { FN(4, 2); }             \
        else if (f_T == 2 && f_KI == 8) { FN(8, 2); }             \
        else if (f_T == 2) { FN(16, 2); }                         \
        else if (f_T == 4 && f_KI == 4) { FN(4, 4); }             \
        else if (f_T == 4 && f_KI == 8) { FN(8, 4); }             \
        else if (f_T == 4) { FN(16, 4); }                         \
        else if (f_KI == 4) { FN(4, 8); }                         \
        else if (f_KI == 8) { FN(8, 8); }                         \
        else { FN(16, 8); }                                       \
    } while (0)
    void set_fused_attr() {
        if (f_team) {
#define BIOEN_SET_ATTR(KI_, T_) set_team_attr<KI_, T_>()
            BIOEN_TEAM_DISPATCH(BIOEN_SET_ATTR);
#undef BIOEN_SET_ATTR
            return;
        }
    }
    template <int KIND>
    void launch_fused(const double* bvec, const double* s0, const double* s1, double* xout, double theta_arg = -1.0) {
        const bool timed = pass_timing && pass_ev_used + 2 <= pass_ev.size();
        if (timed) CUDA_CHECK(cudaEventRecord(pass_ev[pass_ev_used++], stream));
        {
            TeamArgs a{};
            a.Yt = Yt.p; a.ldt = ldt; a.M = M; a.N = N; a.C = f_C; a.stages = f_stages; a.nslab = f_nslab;
            a.chunk = f_chunk; a.ab = ab.p; a.b = bvec; a.s0 = s0; a.s1 = s1; a.theta = theta_arg >= 0.0 ? theta_arg : theta; a.xout = xout;
            a.part = fpart.p; a.ldp = Mpad; a.lse = flse.p; a.evict_first = evict_first;
#define BIOEN_LAUNCH_TEAM(KI_, T_) fused_team_pass<KI_, T_, KIND><<<f_grid, kTThreads, f_smem, stream>>>(a)
            BIOEN_TEAM_DISPATCH(BIOEN_LAUNCH_TEAM);
#undef BIOEN_LAUNCH_TEAM
        }
        if (timed) CUDA_CHECK(cudaEventRecord(pass_ev[pass_ev_used++], stream));
        CUDA_CHECK(cudaGetLastError());
        ++passes_launched;
        ++kernels_launched;
    }
    void merge_fused_rows(bool scaled, int ntail) {
        k_fused_merge_rows<<<(M + 31) / 32, 256, 0, stream>>>(
            M, f_rows, fpart.p, Mpad, scaled ? flse.p : nullptr, lse_pairs(), nranks, msum.p);
        ++kernels_launched;
        if (nranks > 1) comm->allreduce_sum(msum.p, M + ntail, stream);
    }
    void forces_eval_fused_f(double* x, const double* xp, const double* d, double stp) {
        NvtxRange nvtx("bioen:forces_eval_f(fused)");
        {
            ForcesUpdateArgs a{M, x, xp, d, stp, ab.p, sc.p};
            k_forces_update<<<1, 1024, 0, stream>>>(a);
            ++kernels_launched;
        }
        launch_fused<kFusedSoftmaxAvg>(nullptr, Gv.p, nullptr, aux_n.p);   // x_j, CTA-local softmax, avg partials
        const bool xfused = fuse_exchange_forces();
        if (xfused) {
            k_forces_lse_gather<<<1, 256, 0, stream>>>(f_rows, flse.p, sc.p + SC_LSE_MAX, lse_all.p, p2p_dev_raw());
            ++kernels_launched;
        } else {
            k_fused_lse_merge<<<1, 256, 0, stream>>>(f_rows, flse.p, sc.p + SC_LSE_MAX);
            ++kernels_launched;
            gather_lse();
        }
        {
            ForcesWeightsArgs a{};
            a.n = N; a.x = aux_n.p; a.w0 = Gv.p; a.w = w.p; a.lr = aux_n2.p; a.lse_pairs = lse_pairs();
            a.nranks = nranks; a.msum_tail = msum.p + M; a.partials = red_partials.p; a.ticket = ticket.p;
            a.sc = sc.p;
            k_forces_weights<<<vec_blocks_n, kVecThreads, 0, stream>>>(a);
            ++kernels_launched;
        }
        if (xfused) {
            rows_finish(true, 1, false, nullptr, nullptr);
            return;
        }
        merge_fused_rows(true, 1);
        finalize_rows_from_msum(true, false);
    }
    // sharded fused forces path: exchanges issued inside the producing kernels (needs the peer-memory path)
    bool fuse_exchange_forces() const {
        return nranks > 1 && comm && comm->fused_ok((size_t)M + 8) && options.fuse_allowed;
    }
    P2PDev p2p_dev_raw() const { ++comm->exchanges; return comm->dev_args(); }
    void rows_finish(bool scaled, int ntail, bool gradient, double* grad, const double* ddir) {
        RowsFinishArgs a{};
        a.m = M; a.nrows = f_rows; a.part = fpart.p; a.ldp = Mpad; a.lse_rows = scaled ? flse.p : nullptr;
        a.lse_pairs = lse_pairs(); a.nranks = nranks; a.out = msum.p; a.ntail = ntail; a.gradient = gradient ? 1 : 0;
        a.Y = Yobs.p; a.ab = ab.p; a.avg = avg.p; a.theta = theta; a.d = ddir; a.grad = grad;
        a.ticket = ticket.p; a.sc = sc.p; a.p2p = p2p_dev_raw();
        k_forces_rows_finish<<<(M + 31) / 32, 256, 0, stream>>>(a);
        ++kernels_launched;
    }
    void forces_eval_fused_g(double* grad, const double* ddir) {
        NvtxRange nvtx("bioen:forces_eval_g(fused)");
        launch_fused<kFusedGradient>(avg.p, w.p, aux_n2.p, nullptr);       // t_j, E_j, grad partials
        if (fuse_exchange_forces()) {
            rows_finish(false, 0, true, grad, ddir);
            return;
        }
        merge_fused_rows(false, 0);
        {
            ForcesGradArgs a{};
            a.m = M; a.partial = nullptr; a.ld = Mpad; a.L = nCB; a.chunk = chunk; a.msum = msum.p;
            a.d = ddir; a.grad = grad; a.sc = sc.p;
            k_forces_grad<<<1, 1024, 0, stream>>>(a);
            ++kernels_launched;
        }
    }
    // k_finalize_rows on an msum that is already slot-, CTA- and rank-reduced
    void finalize_rows_from_msum(bool is_forces, bool ab_with_avg) {
        FinalizeArgs a{};
        a.m = M; a.partial = nullptr; a.ld = Mpad; a.L = nCB; a.chunk = chunk; a.msum = msum.p;
        a.Y = Yobs.p; a.ab = ab.p; a.avg = avg.p; a.ab_with_avg = ab_with_avg ? 1 : 0;
        a.is_forces = is_forces ? 1 : 0; a.theta = theta;
        a.partials = red_partials.p; a.ticket = ticket.p; a.sc = sc.p;
        a.tail = msum.p + M;
        k_finalize_rows<<<(M + kVecThreads - 1) / kVecThreads, kVecThreads, 0, stream>>>(a);
        ++kernels_launched;
    }

    // exchanges between the ranks inside one f+g evaluation (reported by bench.py)
    int exchanges_per_eval(bool forces) const {
        if (nranks <= 1) return 0;
        if (!forces && fuse_exchange()) return 2;   // M+5 doubles (objective half) + 4 scalars (gradient half)
        return 3;   // forces: (max, sum) gather + avg/KL sum + gradient sum (inside the producing kernels when fused)   // (max, sum) gather + M-vector sum + {3 scalars | gradient M-vector}
    }
    // Sharded log-weights evaluation with the exchanges inside the producing kernels (peer-memory path only): the
    // normalisation pair travels with the row sums, so the objective half needs ONE exchange and no exchange launch.
    bool fuse_exchange() const {
        return nranks > 1 && comm && comm->fused_ok((size_t)M + 5) && options.fuse_allowed;
    }
    P2PDev p2p_dev() const {
        if (nranks > 1 && comm && fuse_exchange()) { ++comm->exchanges; return comm->dev_args(); }
        P2PDev d{};
        d.nranks = 1;
        return d;
    }

    // ---- kernel launch helpers ---------------------------------------------------------------------
    const double* lse_pairs() const { return nranks > 1 ? lse_all.p : sc.p + SC_LSE_MAX; }

    void launch_lse(double* x, const double* xp, const double* d, double stp, const double* w0, bool from_col) {
        LseArgs a{};
        a.n = N; a.x = x; a.xp = xp; a.d = d; a.stp = stp; a.w0 = w0;
        a.col_partial = from_col ? partialB.p : nullptr;
        a.col_ld = Npad; a.col_L = nRT; a.col_chunk = col_chunk();
        a.write_xnorm = from_col ? 0 : 1;
        a.partials = red_partials.p; a.ticket = ticket.p; a.sc = sc.p;
        k_update_lse<<<vec_blocks_n, kVecThreads, 0, stream>>>(a);
        ++kernels_launched;
    }
    void gather_lse() {
        if (nranks > 1) comm->allgather(sc.p + SC_LSE_MAX, lse_all.p, 2, stream);
    }
    template <int MODE, bool SUB>
    void launch_pass(const double* vN, const double* vMb) {
        PassArgs a{};
        a.nRT = nRT; a.nCB = nCB; a.T = T; a.chunk = chunk;
        a.interleave = (MODE == kColPass && interleave_col) ? 1 : 0;
        a.evict_first = evict_first;
        a.vN = vN; a.vMb = vMb; a.ab = ab.p;
        a.partial = (MODE == kRowPass) ? partialA.p : partialB.p;
        a.ld = (MODE == kRowPass) ? Mpad : Npad;
        require_row_major("this evaluation path (tile kernels)");
        if (!has_matrix()) throw std::logic_error("bioen_b200: yTilde has not been uploaded");
        const bool timed = pass_timing && pass_ev_used + 2 <= pass_ev.size();
        if (timed) CUDA_CHECK(cudaEventRecord(pass_ev[pass_ev_used++], stream));
        if (storage_fp32)
            stream_pass_kernel<MODE, SUB, float><<<grid, kPassThreads, kPassSmemBytesF32, stream>>>(tmap, a);
        else
            stream_pass_kernel<MODE, SUB, double><<<grid, kPassThreads, kPassSmemBytes, stream>>>(tmap, a);
        if (timed) CUDA_CHECK(cudaEventRecord(pass_ev[pass_ev_used++], stream));
        CUDA_CHECK(cudaGetLastError());
        ++passes_launched;
        ++kernels_launched;
    }
    // per-launch CUDA-event timing of the matrix passes (bench.py roofline): events bracket every pass kernel
    // on this stream between begin_pass_timing() and end_pass_timing(), which returns the mean duration in ms
    std::vector<cudaEvent_t> pass_ev;
    size_t pass_ev_used = 0;
    bool pass_timing = false;
    void begin_pass_timing(int max_passes) {
        while (pass_ev.size() < (size_t)max_passes * 2) {
            cudaEvent_t e;
            CUDA_CHECK(cudaEventCreate(&e));
            pass_ev.push_back(e);
        }
        pass_ev_used = 0;
        pass_timing = true;
    }
    float end_pass_timing() {
        pass_timing = false;
        sync();
        double total = 0.0;
        size_t cnt = 0;
        for (size_t i = 0; i + 1 < pass_ev_used; i += 2) {
            float t = 0.f;
            CUDA_CHECK(cudaEventElapsedTime(&t, pass_ev[i], pass_ev[i + 1]));
            total += t;
            ++cnt;
        }
        return cnt ? (float)(total / (double)cnt) : 0.f;
    }
    // finish a row pass that produced avg (logw: tail = 3 weighted sums, forces: tail = KL)
    void finalize_rows(bool is_forces, int ntail, bool ab_with_avg) {
        FinalizeArgs a{};
        a.m = M; a.partial = partialA.p; a.ld = Mpad; a.L = nCB; a.chunk = chunk;
        a.Y = Yobs.p; a.ab = ab.p; a.avg = avg.p; a.ab_with_avg = ab_with_avg ? 1 : 0;
        a.is_forces = is_forces ? 1 : 0; a.theta = theta;
        a.partials = red_partials.p; a.ticket = ticket.p; a.sc = sc.p;
        a.tail = msum.p + M;
        if (nranks > 1) {
            k_reduce_row_slots<<<vec_blocks_m, kVecThreads, 0, stream>>>(M, partialA.p, Mpad, nCB, chunk, msum.p);
            ++kernels_launched;
            comm->allreduce_sum(msum.p, M + ntail, stream);
            a.msum = msum.p;
        }
        k_finalize_rows<<<(M + kVecThreads - 1) / kVecThreads, kVecThreads, 0, stream>>>(a);
        ++kernels_launched;
    }

    // ---- persistent cooperative evaluation (persistent_eval.cuh) ------------------------------------------------
    // One kernel per evaluation (or per half).  Used when the matrix is small enough that launch gaps and kernel
    // ramp-up / tail are a visible share of an evaluation.  Auto threshold 0.6 GB per GPU, measured at M = 1000 after
    // the stand-alone path got the interleaved column pass with the gradient epilogue: 0.4 GB 0.1539 vs 0.1652 ms
    // (persistent wins), 1 GB 0.3351 vs 0.3319, 2 GB 0.6262 vs 0.6127, 4 GB 1.1869 vs 1.1670 (stand-alone wins);
    // sharded over 2 GPUs the same: 0.4 GB per GPU 0.1674 vs 0.1815, 1 GB 0.3539 vs 0.3446, 2 GB 0.6423 vs 0.6281;
    // the stand-alone kernels remain the path for large matrices, for the fused two-pass forces kernels and for
    // in-process groups (two cooperative grids cannot be co-resident on one device).
    // slice_eval.cuh: the matrix dealt column-wise into the CTAs' shared memory, 1 grid barrier per evaluation.  Takes
    // precedence over the persistent kernel AND over the fused two-pass forces kernels whenever the problem is small
    // enough (slice_plan); BIOEN_B200_OPT_PERSISTENT = 0 (stand-alone kernels) switches it off as well.
    bool slice_ok() const {
        return slice_pl.ok && slice_coop && options.slice_mode != 0 && options.persistent_mode != 0 && nranks == 1 &&
               Y != nullptr && !storage_fp32 && (ld % 2) == 0 && ld >= N && (reinterpret_cast<uintptr_t>(Y) & 15) == 0;
    }
    void launch_slice(int method, int mode, double* x, const double* xp, const double* d, double stp,
                      double* grad, const double* ddir) {
        SliceArgs a{};
        a.method = method; a.mode = mode; a.M = M; a.N = N;
        a.nc = slice_pl.nc; a.ncs = slice_pl.ncs; a.ms = slice_pl.ms;
        a.cx_log2 = slice_pl.cx_log2; a.l_log2 = slice_pl.l_log2; a.lt_log2 = slice_pl.lt_log2;
        a.Y = Y; a.ld = ld;
        a.x = x; a.xp = xp; a.d = d; a.stp = stp;
        a.Gv = Gv.p; a.w = w.p; a.aux_n = aux_n.p; a.aux_n2 = aux_n2.p; a.grad = grad; a.ddir = ddir;
        a.Yobs = Yobs.p; a.ab = ab.p; a.avg = avg.p; a.theta = theta; a.sc = sc.p;
        a.tab = slice_tab.p; a.gtab = slice_gtab.p; a.part = slice_part.p; a.bar = pe_bar.p; a.ticket = ticket.p;
        // algorithmic passes of the evaluation (the kernel reads the matrix once).  No per-pass events here: a launch is
        // a whole evaluation of ~20 us, and two timing events around it cost a visible share of that.
        const int npass = method == 0 ? (mode == kPEvalBoth ? 2 : 1) : (mode == kPEvalBoth ? 4 : 2);
        void* args[] = {(void*)&a};
        CUDA_CHECK(cudaLaunchCooperativeKernel((const void*)slice_eval_kernel, dim3(slice_pl.grid), dim3(kSliceThreads),
                                               args, slice_pl.smem, stream));
        passes_launched += npass;
        ++kernels_launched;
        ++persistent_launches;
        ++slice_launches;
    }
    bool persistent_for(bool forces) const {
        if (slice_ok()) return true;
        if (!coop_ok || options.persistent_mode == 0 || !has_matrix()) return false;
        if (options.persistent_mode < 0 && matrix_bytes() > kPersistentMaxBytes) return false;
        if (forces) return nranks == 1 && !forces_fused_now();
        if (nranks > 1) return fuse_exchange() && !comm->is_local();
        return true;
    }
    void launch_persistent(int method, int mode, double* x, const double* xp, const double* d, double stp,
                           double* grad, const double* ddir) {
        if (!has_matrix()) throw std::logic_error("bioen_b200: yTilde has not been uploaded");
        if (slice_ok()) {
            launch_slice(method, mode, x, xp, d, stp, grad, ddir);
            return;
        }
        PEvalArgs a{};
        a.method = method; a.mode = mode; a.M = M; a.N = N;
        a.row.nRT = nRT; a.row.nCB = nCB; a.row.T = T; a.row.chunk = chunk; a.row.interleave = 0;
        a.row.evict_first = evict_first; a.row.partial = partialA.p; a.row.ld = Mpad;
        a.col = a.row;
        a.col.partial = partialB.p; a.col.ld = Npad;
        a.x = x; a.xp = xp; a.d = d; a.stp = stp;
        a.Gv = Gv.p; a.w = w.p; a.aux_n = aux_n.p; a.aux_n2 = aux_n2.p; a.grad = grad; a.ddir = ddir;
        a.Yobs = Yobs.p; a.ab = ab.p; a.avg = avg.p; a.msum = msum.p; a.theta = theta; a.sc = sc.p;
        a.part = pe_part.p; a.bar = pe_bar.p; a.ticket = ticket.p;
        if (method == 0 && nranks > 1) a.p2p = p2p_dev(); else a.p2p.nranks = 1;
        // The kernel's passes and their readers use the contiguous tile order for both passes: dealing the column
        // pass's runs round-robin, as the stand-alone kernel does, measured 150.2 us vs 149.1 us contiguous at config 2
        // (0.4 GB) -- no gain for the matrix sizes this kernel is used for.
        // No per-launch events: a launch is a whole evaluation, so the callers that time evaluations
        // (bioen_b200_time_evals) derive the per-pass figure from the step time instead of paying two timing events
        // per launch inside the timed region.  Cooperative launch = the driver's guarantee that all CTAs are resident
        // (the grid barriers need it).
        const int npass = method == 0 ? (mode == kPEvalBoth ? 2 : 1) : (mode == kPEvalBoth ? 4 : 2);
        void* args[] = {(void*)&tmap, (void*)&a};
        const void* fn = storage_fp32 ? (const void*)persistent_eval_kernel<float>
                                      : (const void*)persistent_eval_kernel<double>;
        CUDA_CHECK(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(kPEvalThreads), args,
                                               (size_t)(storage_fp32 ? kPassSmemBytesF32 : kPassSmemBytes), stream));
        passes_launched += npass;
        ++kernels_launched;
        ++persistent_launches;
    }

    // ---- log-weights evaluation (c_bioen_kernels_logw.c:525-561) ------------------------------------------
    // x (device, N): evaluated point; when xp != nullptr it is first formed as xp + stp*d.
    // grad == nullptr -> objective only (one pass over Y).  ddir: optional direction for sc[SC_DG].
    // The evaluation is split at the point where the objective is complete: logw_eval_f leaves w, avg and the
    // residuals on the device, logw_eval_g adds the gradient of that same point (callers that learn from f alone
    // that the gradient is not needed -- a backtracking trial that fails the Armijo test, GSL's f-then-df pattern --
    // skip or defer the second pass over Y).  eval_gen changes with every objective evaluation.
    long long eval_gen = 0;
    void logw_eval(double* x, const double* xp, const double* d, double stp, double* grad, const double* ddir) {
        if (grad && persistent_for(false)) {
            NvtxRange nvtx("bioen:logw_eval(persistent)");
            if (!have_logw) throw std::logic_error("bioen_b200: log-weights data not set");
            ++eval_gen;
            launch_persistent(0, kPEvalBoth, x, xp, d, stp, grad, ddir);
            eval_fused = false;
            return;
        }
        logw_eval_f(x, xp, d, stp);
        if (grad) logw_eval_g(x, grad, ddir);
    }
    void logw_eval_f(double* x, const double* xp, const double* d, double stp) {
        NvtxRange nvtx("bioen:logw_eval_f");
        if (!have_logw) throw std::logic_error("bioen_b200: log-weights data not set");
        ++eval_gen;
        if (persistent_for(false)) {
            launch_persistent(0, kPEvalObjective, x, xp, d, stp, nullptr, nullptr);
            eval_fused = nranks > 1;
            return;
        }
        launch_lse(x, xp, d, stp, nullptr, false);
        const bool fused = fuse_exchange();
        eval_fused = fused;
        if (!fused) gather_lse();
        {
            LogwWeightsArgs a{};
            a.n = N; a.g = x; a.G = Gv.p; a.w = w.p; a.lse_pairs = lse_pairs(); a.nranks = nranks;
            a.msum_tail = msum.p + M; a.partials = red_partials.p; a.ticket = ticket.p; a.sc = sc.p;
            a.local_only = fused ? 1 : 0;
            k_logw_weights<<<vec_blocks_n, kVecThreads, 0, stream>>>(a);
            ++kernels_launched;
        }
        launch_pass<kRowPass, false>(w.p, nullptr);
        if (fused) {
            RowsExchangeArgs a{};
            a.m = M; a.partial = partialA.p; a.ld = Mpad; a.L = nCB; a.chunk = chunk; a.msum = msum.p;
            a.p2p = p2p_dev(); a.Y = Yobs.p; a.ab = ab.p; a.avg = avg.p; a.theta = theta; a.sc = sc.p;
            k_logw_rows_exchange_finalize<<<1, kRowsXThreads, 0, stream>>>(a);
            ++kernels_launched;
        } else {
            finalize_rows(false, 3, true);
        }
    }
    // will logw_eval_g form the gradient inside the column pass (and so stream it out while the pass runs)?
    bool colgrad_eligible() const {
        return (nranks == 1 || fuse_exchange()) && interleave_col && !persistent_for(false);
    }
    bool eval_fused = false;   // the last logw_eval_f left un-normalised e_j in `w` (fused sharded path)
    void logw_eval_g(const double* x, double* grad, const double* ddir) {
        NvtxRange nvtx("bioen:logw_eval_g");
        if (persistent_for(false) && (nranks == 1 || eval_fused)) {
            launch_persistent(0, kPEvalGradient, const_cast<double*>(x), nullptr, nullptr, 0.0, grad, ddir);
            eval_fused = false;
            return;
        }
        // single GPU, whole runs per CTA: the column pass forms the gradient itself (stream_colgrad_kernel)
        auto aligned16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
        const bool sharded_fused = nranks > 1 && eval_fused;
        if ((nranks == 1 || sharded_fused) && interleave_col && aligned16(x) && aligned16(grad) &&
            aligned16(Gv.p) && aligned16(w.p)) {
            PassArgs pa{};
            pa.nRT = nRT; pa.nCB = nCB; pa.T = T; pa.chunk = chunk; pa.interleave = 1; pa.evict_first = evict_first;
            pa.ab = ab.p; pa.partial = partialB.p; pa.ld = Npad;
            ColGradArgs ga{};
            ga.n = N; ga.g = x; ga.G = Gv.p; ga.w = w.p; ga.d = ddir; ga.grad = grad; ga.theta = theta; ga.sc = sc.p;
            ga.i_gbar = SC_GBAR; ga.i_Gbar = SC_CAPGBAR; ga.cta_part = colgrad_part.p;
            ga.i_wscale = sharded_fused ? SC_WSCALE : -1;
            ga.wio = w.p;
            const bool timed = pass_timing && pass_ev_used + 2 <= pass_ev.size();
            if (timed) CUDA_CHECK(cudaEventRecord(pass_ev[pass_ev_used++], stream));
            if (storage_fp32)
                stream_colgrad_kernel<float><<<grid, kPassThreads, kPassSmemBytesF32, stream>>>(tmap, pa, ga);
            else
                stream_colgrad_kernel<double><<<grid, kPassThreads, kPassSmemBytes, stream>>>(tmap, pa, ga);
            if (timed) CUDA_CHECK(cudaEventRecord(pass_ev[pass_ev_used++], stream));
            CUDA_CHECK(cudaGetLastError());
            if (sharded_fused) k_colgrad_finish_sharded<<<1, 256, 0, stream>>>(grid, colgrad_part.p, sc.p, p2p_dev());
            else k_colgrad_finish<<<1, 256, 0, stream>>>(grid, colgrad_part.p, sc.p, SC_DG, SC_GNORM2, SC_GINF);
            ++passes_launched;
            kernels_launched += 2;
            eval_fused = false;
            return;
        }
        launch_pass<kColPass, true>(nullptr, nullptr);
        {
            LogwGradArgs a{};
            a.n = N; a.col_partial = partialB.p; a.ld = Npad; a.L = nRT; a.chunk = col_chunk();
            a.g = x; a.G = Gv.p; a.w = w.p; a.d = ddir; a.grad = grad; a.theta = theta;
            a.partials = red_partials.p; a.ticket = ticket.p; a.sc = sc.p;
            a.wio = w.p;
            if (eval_fused) a.p2p = p2p_dev(); else a.p2p.nranks = 1;
            k_logw_grad<<<vec_blocks_n, kVecThreads, 0, stream>>>(a);
            ++kernels_launched;
        }
        if (nranks > 1 && !eval_fused) comm->allreduce_sum(sc.p + SC_DG, 3, stream);  // dg, ||g||^2, ||x||^2
        eval_fused = false;   // `w` is normalised now
    }
    // weights only (the reference's _get_weights): w normalised over all ranks; returns nothing, see sc[]
    void logw_weights_only(double* x) {
        ++eval_gen;
        launch_lse(x, nullptr, nullptr, 0.0, nullptr, false);
        gather_lse();
        LogwWeightsArgs a{};
        a.n = N; a.g = x; a.G = x; a.w = w.p; a.lse_pairs = lse_pairs(); a.nranks = nranks;
        a.msum_tail = msum.p + M; a.partials = red_partials.p; a.ticket = ticket.p; a.sc = sc.p;
        k_logw_weights<<<vec_blocks_n, kVecThreads, 0, stream>>>(a);
        ++kernels_launched;
    }

    // ---- forces evaluation (c_bioen_kernels_forces.c:43-76) ----------------------------------------------
    // x (device, M): forces; formed as xp + stp*d when xp != nullptr.  The M-dimensional state is replicated
    // on every rank.  grad == nullptr -> objective only (two passes over Y).
    void forces_eval(double* x, const double* xp, const double* d, double stp, double* grad, const double* ddir) {
        if (grad && have_forces && persistent_for(true)) {
            NvtxRange nvtx("bioen:forces_eval(persistent)");
            ++eval_gen;
            forces_x = x;
            launch_persistent(1, kPEvalBoth, x, xp, d, stp, grad, ddir);
            return;
        }
        forces_eval_f(x, xp, d, stp);
        if (grad) forces_eval_g(grad, ddir);
    }
    double* forces_x = nullptr;   // the forces vector of the last objective half (persistent gradient half)
    bool forces_fused_now() const { return fused_ready && (options.allow_fused || yt_only); }
    void forces_eval_f(double* x, const double* xp, const double* d, double stp) {
        if (!have_forces) throw std::logic_error("bioen_b200: forces data not set");
        ++eval_gen;
        if (forces_fused_now() && !slice_ok()) {
            forces_eval_fused_f(x, xp, d, stp);
            return;
        }
        if (persistent_for(true)) {
            forces_x = x;
            launch_persistent(1, kPEvalObjective, x, xp, d, stp, nullptr, nullptr);
            return;
        }
        {
            ForcesUpdateArgs a{M, x, xp, d, stp, ab.p, sc.p};
            k_forces_update<<<1, 1024, 0, stream>>>(a);
            ++kernels_launched;
        }
        launch_pass<kColPass, false>(nullptr, nullptr);                 // x_j = sum_i f_i y_ij
        launch_lse(aux_n.p, nullptr, nullptr, 0.0, Gv.p, true);          // assemble x_j, (max, sum w0 e^{x-max})
        gather_lse();
        {
            ForcesWeightsArgs a{};
            a.n = N; a.x = aux_n.p; a.w0 = Gv.p; a.w = w.p; a.lr = aux_n2.p; a.lse_pairs = lse_pairs();
            a.nranks = nranks; a.msum_tail = msum.p + M; a.partials = red_partials.p; a.ticket = ticket.p;
            a.sc = sc.p;
            k_forces_weights<<<vec_blocks_n, kVecThreads, 0, stream>>>(a);
            ++kernels_launched;
        }
        launch_pass<kRowPass, false>(w.p, nullptr);                     // avg_i
        finalize_rows(true, 1, false);                                  // r_i, chi2, f; ab = {r_i, 0}
    }
    // gradient of the point forces_eval_f was last called for
    void forces_eval_g(double* grad, const double* ddir) {
        if (forces_fused_now() && !slice_ok()) {
            forces_eval_fused_g(grad, ddir);
            return;
        }
        if (persistent_for(true)) {
            launch_persistent(1, kPEvalGradient, forces_x, nullptr, nullptr, 0.0, grad, ddir);
            return;
        }
        launch_pass<kColPass, false>(nullptr, nullptr);                 // t_j = sum_i y_ij r_i
        {
            ForcesEArgs a{};
            a.n = N; a.col_partial = partialB.p; a.ld = Npad; a.L = nRT; a.chunk = col_chunk();
            a.w = w.p; a.lr = aux_n2.p; a.E = aux_n.p; a.theta = theta;   // E overwrites x_j (no longer needed)
            k_forces_E<<<vec_blocks_n, kVecThreads, 0, stream>>>(a);
            ++kernels_launched;
        }
        launch_pass<kRowPass, true>(aux_n.p, avg.p);                    // grad_i = sum_j (y_ij - avg_i) E_j
        {
            ForcesGradArgs a{};
            a.m = M; a.partial = partialA.p; a.ld = Mpad; a.L = nCB; a.chunk = chunk;
            a.d = ddir; a.grad = grad; a.sc = sc.p;
            if (nranks > 1) {
                k_reduce_row_slots<<<vec_blocks_m, kVecThreads, 0, stream>>>(M, partialA.p, Mpad, nCB, chunk, msum.p);
                ++kernels_launched;
                comm->allreduce_sum(msum.p, M, stream);
                a.msum = msum.p;
            }
            k_forces_grad<<<1, 1024, 0, stream>>>(a);
            ++kernels_launched;
        }
    }
    // weights only (the reference's _get_weights_from_forces): leaves normalised w in `w`
    void forces_weights_only(double* x) {
        if (!have_forces) throw std::logic_error("bioen_b200: forces data not set");
        if (yt_only) {   // the objective half of the fused path leaves the normalised weights in `w`
            forces_eval_f(x, nullptr, nullptr, 0.0);
            return;
        }
        ++eval_gen;
        ForcesUpdateArgs u{M, x, nullptr, nullptr, 0.0, ab.p, sc.p};
        k_forces_update<<<1, 1024, 0, stream>>>(u);
        launch_pass<kColPass, false>(nullptr, nullptr);
        launch_lse(aux_n.p, nullptr, nullptr, 0.0, Gv.p, true);
        gather_lse();
        ForcesWeightsArgs a{};
        a.n = N; a.x = aux_n.p; a.w0 = Gv.p; a.w = w.p; a.lr = aux_n2.p; a.lse_pairs = lse_pairs();
        a.nranks = nranks; a.msum_tail = msum.p + M; a.partials = red_partials.p; a.ticket = ticket.p;
        a.sc = sc.p;
        k_forces_weights<<<vec_blocks_n, kVecThreads, 0, stream>>>(a);
        kernels_launched += 3;
    }
    // objective (and gradient when grad != nullptr) of the forces method for GIVEN weights already in `w`
    // (reference semantics of _bioen_log_posterior_forces / _grad_bioen_log_posterior_forces,
    // c_bioen_kernels_forces.c:227-340)
    void forces_from_weights(double* grad) {
        require_row_major("the given-weights forces objective");
        ++eval_gen;
        if (!have_forces) throw std::logic_error("bioen_b200: forces data not set");
        {
            ForcesLrArgs a{N, w.p, Gv.p, aux_n2.p, msum.p + M, red_partials.p, ticket.p};
            k_forces_lr_from_w<<<vec_blocks_n, kVecThreads, 0, stream>>>(a);
            ++kernels_launched;
        }
        launch_pass<kRowPass, false>(w.p, nullptr);
        finalize_rows(true, 1, false);
        if (!grad) return;
        launch_pass<kColPass, false>(nullptr, nullptr);
        {
            ForcesEArgs a{};
            a.n = N; a.col_partial = partialB.p; a.ld = Npad; a.L = nRT; a.chunk = col_chunk();
            a.w = w.p; a.lr = aux_n2.p; a.E = aux_n.p; a.theta = theta;
            k_forces_E<<<vec_blocks_n, kVecThreads, 0, stream>>>(a);
            ++kernels_launched;
        }
        launch_pass<kRowPass, true>(aux_n.p, avg.p);
        {
            ForcesGradArgs a{};
            a.m = M; a.partial = partialA.p; a.ld = Mpad; a.L = nCB; a.chunk = chunk;
            a.d = nullptr; a.grad = grad; a.sc = sc.p;
            if (nranks > 1) {
                k_reduce_row_slots<<<vec_blocks_m, kVecThreads, 0, stream>>>(M, partialA.p, Mpad, nCB, chunk, msum.p);
                ++kernels_launched;
                comm->allreduce_sum(msum.p, M, stream);
                a.msum = msum.p;
            }
            k_forces_grad<<<1, 1024, 0, stream>>>(a);
            ++kernels_launched;
        }
    }
    // avg = Y . v for an arbitrary N-vector v already in `w` (post-processing: yopt = y . wopt)
    void average_of_w(double* avg_out_dev) {
        ++eval_gen;
        if (yt_only) {
            // the gradient pass of the fused kernels with r = 0, lr = 0, avg = 0, theta = 1 accumulates
            // sum_j y_ij * ((1 + 0) * 1 + 0) * w_j = (yTilde . w)_i -- one pass over Yt, summed over the ranks
            if (!fused_ready) prepare_fused();
            if (!fused_ready) throw std::logic_error("bioen_b200: structure-major-only mode: fused kernels unavailable");
            aux_n2.ensure(Npad + 8);
            CUDA_CHECK(cudaMemsetAsync(ab.p, 0, (size_t)2 * Mpad * sizeof(double), stream));
            CUDA_CHECK(cudaMemsetAsync(avg.p, 0, (size_t)Mpad * sizeof(double), stream));
            CUDA_CHECK(cudaMemsetAsync(aux_n2.p, 0, (size_t)(Npad + 8) * sizeof(double), stream));
            launch_fused<kFusedGradient>(avg.p, w.p, aux_n2.p, nullptr, 1.0);
            merge_fused_rows(false, 0);
            d2d(avg_out_dev, msum.p, M);
            return;
        }
        launch_pass<kRowPass, false>(w.p, nullptr);
        k_reduce_row_slots<<<vec_blocks_m, kVecThreads, 0, stream>>>(M, partialA.p, Mpad, nCB, chunk, msum.p);
        ++kernels_launched;
        if (nranks > 1) comm->allreduce_sum(msum.p, M, stream);
        d2d(avg_out_dev, msum.p, M);
    }

    // the host reads the scalar file once per line-search trial: spin on an event instead of
    // cudaStreamSynchronize, whose default scheduling may yield the CPU (milliseconds on a busy host)
    cudaEvent_t fetch_ev = nullptr;
    void spin_sync() {
        if (!fetch_ev) CUDA_CHECK(cudaEventCreateWithFlags(&fetch_ev, cudaEventDisableTiming));
        CUDA_CHECK(cudaEventRecord(fetch_ev, stream));
        cudaError_t e;
        while ((e = cudaEventQuery(fetch_ev)) == cudaErrorNotReady) {
        }
        CUDA_CHECK(e);
    }
    // The host reads the scalar file after (almost) every evaluation.  Default: a one-warp kernel stores the 64 doubles
    // straight into the page-locked host copy (mapped under unified addressing), fences at system scope and then
    // stores a sequence number; the host spins on that number.  This replaces a 512-byte copy-engine transfer + event
    // (several microseconds of DMA and driver latency) by posted PCIe writes from an SM -- visible at small problem
    // sizes, where an evaluation takes ~20 us.  BIOEN_B200_OPT_FETCH_ZEROCOPY = 0: the copy.
    unsigned long long fetch_seq = 0;
    void fetch_scalars() {
        NvtxRange nvtx("bioen:fetch_scalars");
        if (!options.fetch_zero_copy) {
            d2h(h_sc, sc.p, SC_COUNT);
            spin_sync();
            return;
        }
        const double seq = (double)(++fetch_seq);
        k_publish_scalars<<<1, 64, 0, stream>>>(sc.p, h_sc, SC_COUNT, h_sc + SC_COUNT + 1, seq);
        CUDA_CHECK(cudaGetLastError());
        volatile double* flag = h_sc + SC_COUNT + 1;
        unsigned long long spins = 0;
        while (*flag != seq) {
            if ((++spins & 0xFFFFF) == 0) {   // every ~1e6 polls: has the stream failed?
                const cudaError_t e = cudaStreamQuery(stream);
                if (e != cudaSuccess && e != cudaErrorNotReady) CUDA_CHECK(e);
                if (e == cudaSuccess && *flag != seq) {   // the kernel is done but the flag did not arrive: fall back
                    d2h(h_sc, sc.p, SC_COUNT);
                    spin_sync();
                    return;
                }
            }
        }
        std::atomic_thread_fence(std::memory_order_acquire);
    }
};

}  // namespace bioen
