// comm.cuh -- multi-GPU plumbing for the N-sharded problem (one process per GPU).
//
// The structure axis N is split across ranks; per evaluation the ranks exchange only O(M) doubles
// (SURVEY.md section 8e).  NCCL is used directly from this library so the collectives are enqueued on the
// same CUDA stream as the kernels, between them, without going back to Python.  libnccl is resolved at run
// time with dlopen: inside a PyTorch process that is the NCCL torch already loaded; a single-GPU user never
// needs NCCL at all.  The communicator is created from a 128-byte unique id that the Python layer
// broadcasts through torch.distributed (bioen_b200/dist.py).
//
// The exchanges are tiny (3 ... M+3 doubles) and sit on the critical path of every evaluation and of every
// L-BFGS dot product, so their cost is pure latency.  NCCL needs ~25-30 us for one; the path therefore carries its
// own exchange over NVLink peer memory (k_p2p_exchange below): every rank owns an inbox that its peers map through
// CUDA IPC, one small kernel stores the rank's contribution straight into every peer's inbox, publishes a
// release-flag, waits for the peers' flags and combines the inboxes in rank order (so all ranks hold bit-identical
// results).  NCCL is kept for the bootstrap (handle exchange), for messages larger than the inbox, and as the
// collective path when peer mapping is not available (BIOEN_B200_P2P=0 forces it).
#pragma once
#include <dlfcn.h>

#include <chrono>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <vector>

#include "common.cuh"

namespace bioen {

struct NcclApi {
    // minimal slice of nccl.h (ABI-stable since NCCL 2.x)
    typedef struct ncclComm* comm_t;
    struct unique_id { char internal[128]; };
    int (*GetUniqueId)(unique_id*) = nullptr;
    int (*CommInitRank)(comm_t*, int, unique_id, int) = nullptr;
    int (*CommDestroy)(comm_t) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, comm_t, cudaStream_t) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, comm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    void* handle = nullptr;
    static constexpr int kFloat64 = 8;  // ncclDouble
    static constexpr int kSum = 0;      // ncclSum
    static constexpr int kMax = 2;      // ncclMax

    static NcclApi& get() {
        static NcclApi api;
        if (!api.handle) {
            const char* names[] = {"libnccl.so.2", "libnccl.so"};
            for (const char* nm : names) {
                api.handle = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
                if (api.handle) break;
            }
            if (!api.handle) throw std::runtime_error("bioen_b200: cannot dlopen libnccl.so.2 (multi-GPU path)");
            auto sym = [&](const char* s) {
                void* p = dlsym(api.handle, s);
                if (!p) throw std::runtime_error(std::string("bioen_b200: missing NCCL symbol ") + s);
                return p;
            };
            api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
            api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
            api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
            api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(sym("ncclAllReduce"));
            api.AllGather = reinterpret_cast<decltype(api.AllGather)>(sym("ncclAllGather"));
            api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
        }
        return api;
    }
};

// ---- peer-memory exchange ---------------------------------------------------------------------------------
// Region owned by each rank (one cudaMalloc, mapped by every peer):
//   [0, 128)    flags[src]  last epoch whose contribution rank `src` has delivered here (monotonic)
//   [128, 136)  epoch       this rank's exchange counter (device side)
//   [256, ...)  inbox[2][nranks][cap] doubles, indexed by epoch parity and source rank
// Parity double buffering is enough: a rank can start exchange e+2 only after every peer has published e+1,
// i.e. after every peer has finished reading exchange e.
constexpr int kP2PMaxRanks = 16;
constexpr int kP2PThreads = 1024;
constexpr size_t kP2PHeaderBytes = 256;
constexpr size_t kP2PMaxCount = 8192;  // doubles per rank and exchange; larger messages go through NCCL
enum P2POp { kP2PSum = 0, kP2PMax = 1, kP2PGather = 2 };

// what a kernel needs to take part in an exchange (passed by value inside the kernel arguments); nranks <= 1 = off
struct P2PDev {
    unsigned char* region[kP2PMaxRanks];  // region[r]: rank r's region as mapped in this process
    int rank, nranks;
    long long cap;
    unsigned long long timeout_ns;
    int ll;   // 1: flag-in-data ("LL") delivery, 0: data + fence + flag
};

struct P2PArgs {
    P2PDev dev;
    const double* send;
    double* recv;
    int count, op;
};

__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// One exchange, executed by ALL threads of ONE block (a 1-block kernel, or the block of a larger kernel that
// finishes its grid reduction -- the producers of the exchanged values call this from their last-arriving block, so
// an evaluation needs no separate exchange launches).  Delivers send[0..count) into every rank's inbox and returns
// a pointer to this rank's inbox of the current epoch: rank r's contribution is at inbox + r*cap.  The caller
// combines the contributions itself (in rank order: all ranks get bit-identical results) and must not start the
// NEXT exchange before it has finished reading (guaranteed by stream order / by being the same block).
// *fail is set when a peer did not arrive within the timeout (the caller poisons its result with NaN).
__device__ __forceinline__ const double* p2p_deliver_and_wait_fenced(const P2PDev& a, const double* send, int count,
                                                                     int* fail) {
    __shared__ unsigned long long s_epoch;
    __shared__ int s_fail;
    unsigned char* me = a.region[a.rank];
    const int tid = threadIdx.x, nthr = blockDim.x, R = a.nranks;
    __syncthreads();   // `send` may have been produced by other threads of this block
    if (tid == 0) {
        unsigned long long* ep = reinterpret_cast<unsigned long long*>(me + 128);
        s_epoch = *ep + 1;
        *ep = s_epoch;
        s_fail = 0;
    }
    __syncthreads();
    const unsigned long long epoch = s_epoch;
    const size_t par = (size_t)(epoch & 1);
    // Read each value ONCE (up to four independent loads in flight per thread), then store it to every inbox.  A loop
    // "for every rank: dst[i] = send[i]" re-reads send[] per rank, and because dst may alias send the compiler keeps
    // every load behind the previous store: R x count/nthr serialised L2 round trips (measured: 19.7 us of a 1005-double
    // exchange between 2 ranks; the same exchange takes ~5 us this way).
    const size_t slot = (par * R + a.rank) * a.cap;
    for (int i0 = tid; i0 < count; i0 += 4 * nthr) {
        double v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * nthr;
            v[u] = i < count ? send[i] : 0.0;
        }
        for (int r = 0; r < R; ++r) {
            double* dst = reinterpret_cast<double*>(a.region[r] + kP2PHeaderBytes) + slot;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = i0 + u * nthr;
                if (i < count) dst[i] = v[u];
            }
        }
    }
    __threadfence_system();
    __syncthreads();
    if (tid < R) {
        st_release_sys(reinterpret_cast<unsigned long long*>(a.region[tid]) + a.rank, epoch);
        const unsigned long long* flag = reinterpret_cast<const unsigned long long*>(me) + tid;
        const unsigned long long t0 = global_timer_ns();
        while (ld_acquire_sys(flag) < epoch) {
            if (global_timer_ns() - t0 > a.timeout_ns) {  // a peer never arrived: poison the result, do not hang
                s_fail = 1;
                break;
            }
        }
    }
    __syncthreads();
    *fail = s_fail;
    return reinterpret_cast<const double*>(me + kP2PHeaderBytes) + par * R * a.cap;
}

// The same exchange with the flag travelling INSIDE the data (the idea of NCCL's LL protocol): every double is sent
// as one 16-byte cell {lo32 | epoch32 << 32, hi32 | epoch32 << 32}; each 8-byte half is written atomically, so a
// receiver that sees the current epoch in both halves has the value -- no system-wide fence after the stores, no
// separate flag store, no flag poll: one NVLink one-way latency instead of store + fence round trip + flag.  The
// received values are unpacked into the plain inbox so callers read them exactly as in the fenced variant.
// Region: the LL cells live behind the plain inbox ([2][R][cap] doubles), [2][R][cap] cells of 16 bytes.
__device__ __forceinline__ const double* p2p_deliver_and_wait_ll(const P2PDev& a, const double* send, int count,
                                                                 int* fail) {
    __shared__ unsigned long long s_epoch;
    __shared__ int s_fail;
    unsigned char* me = a.region[a.rank];
    const int tid = threadIdx.x, nthr = blockDim.x, R = a.nranks;
    __syncthreads();   // `send` may have been produced by other threads of this block
    if (tid == 0) {
        unsigned long long* ep = reinterpret_cast<unsigned long long*>(me + 128);
        s_epoch = *ep + 1;
        *ep = s_epoch;
        s_fail = 0;
    }
    __syncthreads();
    const unsigned long long epoch = s_epoch;
    const unsigned long long tag = (epoch & 0xffffffffull) << 32;
    const size_t par = (size_t)(epoch & 1);
    const size_t plain_bytes = (size_t)2 * R * a.cap * sizeof(double);
    const size_t slot = (par * R + a.rank) * a.cap;
    for (int i0 = tid; i0 < count; i0 += 4 * nthr) {
        unsigned long long lo[4], hi[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * nthr;
            const unsigned long long bits = (unsigned long long)__double_as_longlong(i < count ? send[i] : 0.0);
            lo[u] = (bits & 0xffffffffull) | tag;
            hi[u] = (bits >> 32) | tag;
        }
        for (int r = 0; r < R; ++r) {
            ulonglong2* dst = reinterpret_cast<ulonglong2*>(a.region[r] + kP2PHeaderBytes + plain_bytes) + slot;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = i0 + u * nthr;
                if (i < count)
                    asm volatile("st.volatile.global.v2.u64 [%0], {%1, %2};" ::"l"(dst + i), "l"(lo[u]), "l"(hi[u])
                                 : "memory");
            }
        }
    }
    // receive: every cell of every rank, unpacked into the plain inbox
    double* plain = reinterpret_cast<double*>(me + kP2PHeaderBytes) + par * R * a.cap;
    const ulonglong2* cells = reinterpret_cast<const ulonglong2*>(me + kP2PHeaderBytes + plain_bytes) + par * R * a.cap;
    const unsigned long long t0 = global_timer_ns();
    bool bad = false;
    for (int r = 0; r < R && !bad; ++r) {
        for (int i = tid; i < count; i += nthr) {
            unsigned long long x, y;
            unsigned int spins = 0;
            for (;;) {
                asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(x), "=l"(y) : "l"(cells + r * a.cap + i)
                             : "memory");
                if ((x & 0xffffffff00000000ull) == tag && (y & 0xffffffff00000000ull) == tag) break;
                if ((++spins & 1023u) == 0 && global_timer_ns() - t0 > a.timeout_ns) { bad = true; break; }
            }
            if (bad) break;
            plain[r * a.cap + i] = __longlong_as_double((long long)((x & 0xffffffffull) | (y << 32)));
        }
    }
    if (bad) s_fail = 1;
    __syncthreads();
    *fail = s_fail;
    return plain;
}

__device__ __forceinline__ const double* p2p_deliver_and_wait(const P2PDev& a, const double* send, int count,
                                                              int* fail) {
    return a.ll ? p2p_deliver_and_wait_ll(a, send, count, fail) : p2p_deliver_and_wait_fenced(a, send, count, fail);
}

__device__ __forceinline__ double p2p_nan() { return __longlong_as_double(0x7ff8000000000000LL); }

// exchange + the standard combinations (sum / max / gather), all threads of one block
__device__ __forceinline__ void p2p_exchange_block(const P2PDev& a, const double* send, double* recv, int count,
                                                   int op) {
    int fail;
    const double* in = p2p_deliver_and_wait(a, send, count, &fail);
    const int tid = threadIdx.x, nthr = blockDim.x, R = a.nranks;
    if (fail) {
        const int total = (op == kP2PGather) ? count * R : count;
        for (int i = tid; i < total; i += nthr) recv[i] = p2p_nan();
    } else if (op == kP2PGather) {
        for (int r = 0; r < R; ++r)
            for (int i = tid; i < count; i += nthr) recv[(size_t)r * count + i] = __ldcg(in + r * a.cap + i);
    } else {
        for (int i = tid; i < count; i += nthr) {
            double s = __ldcg(in + i);
            for (int r = 1; r < R; ++r) {
                const double v = __ldcg(in + r * a.cap + i);
                s = (op == kP2PSum) ? s + v : fmax(s, v);
            }
            recv[i] = s;
        }
    }
    __syncthreads();
}

__global__ void __launch_bounds__(kP2PThreads, 1) k_p2p_exchange(const P2PArgs a) {
    p2p_exchange_block(a.dev, a.send, a.recv, a.count, a.op);
}

// ---- in-process groups ------------------------------------------------------------------------------------
// Several contexts of ONE process (one host thread each; the same or different devices) form a group without
// NCCL or CUDA IPC: every rank publishes its region pointer in a process-wide table and waits for the others.
// This is how the sharded path -- the exchange protocol and the rank-local arithmetic -- is exercised on a box
// with a single GPU (tests/test_gpu_loopback.py); with one GPU per rank it also serves single-process multi-GPU use.
struct LocalGroup {
    std::mutex mu;
    std::condition_variable cv;
    int nranks = 0, published = 0, closed = 0;
    unsigned char* region[kP2PMaxRanks] = {};
    int device[kP2PMaxRanks] = {};
};
inline LocalGroup& local_group(int id) {
    static std::mutex mu;
    static std::map<int, LocalGroup> groups;
    std::lock_guard<std::mutex> lk(mu);
    return groups[id];
}

class Comm {
   public:
    int rank = 0, nranks = 1;
    NcclApi::comm_t comm = nullptr;
    // peer-memory exchange state
    bool p2p = false;         // regions mapped on every rank
    bool use_p2p = true;      // run-time switch (BIOEN_B200_OPT_P2P); must be flipped on all ranks together
    unsigned char* region = nullptr;
    unsigned char* mapped[kP2PMaxRanks] = {};
    long long cap = 0;
    long long p2p_launches = 0;
    bool use_ll = true;       // flag-in-data delivery (BIOEN_B200_EXCHANGE_LL=0 selects data + fence + flag)
    int local_group_id = -1;  // >= 0: in-process group (no NCCL, no IPC)
    unsigned long long timeout_ns = 120ull * 1000000000ull;  // generous: ranks may be skewed by host-side setup

    static void unique_id(char out[128]) {
        NcclApi::unique_id id;
        check(NcclApi::get().GetUniqueId(&id), "ncclGetUniqueId");
        memcpy(out, id.internal, 128);
    }
    Comm(const char id_bytes[128], int rank_, int nranks_) : rank(rank_), nranks(nranks_) {
        NcclApi::unique_id id;
        memcpy(id.internal, id_bytes, 128);
        check(NcclApi::get().CommInitRank(&comm, nranks, id, rank), "ncclCommInitRank");
    }
    // in-process group: rank `rank_` of `nranks_` contexts of this process that pass the same group id
    Comm(int group_id, int rank_, int nranks_) : rank(rank_), nranks(nranks_), local_group_id(group_id) {
        if (group_id < 0) throw std::invalid_argument("bioen_b200: local group id must be >= 0");
        if (nranks_ > kP2PMaxRanks) throw std::invalid_argument("bioen_b200: too many ranks for a local group");
    }
    ~Comm() {
        release_p2p();
        if (comm) NcclApi::get().CommDestroy(comm);
    }
    bool is_local() const { return local_group_id >= 0; }
    void read_timeout_env() {
        if (const char* e = getenv("BIOEN_B200_P2P_TIMEOUT_S")) {
            const double sec = atof(e);
            if (sec > 0) timeout_ns = (unsigned long long)(sec * 1e9);
        }
        if (const char* e = getenv("BIOEN_B200_EXCHANGE_LL")) use_ll = e[0] != '0';
    }
    // what the producing kernels need to run an exchange themselves; nranks = 1 switches their exchange code off
    P2PDev dev_args() const {
        P2PDev d{};
        d.rank = rank; d.nranks = (p2p && use_p2p) ? nranks : 1; d.cap = cap; d.timeout_ns = timeout_ns;
        d.ll = use_ll ? 1 : 0;
        for (int r = 0; r < nranks && r < kP2PMaxRanks; ++r) d.region[r] = mapped[r];
        return d;
    }
    bool fused_ok(size_t count) const { return p2p && use_p2p && count <= (size_t)cap; }
    // publish this rank's region in the process-wide table and wait for the rest of the group
    void enable_local(long long cap_doubles, int device) {
        read_timeout_env();
        cap = cap_doubles;
        const size_t bytes = kP2PHeaderBytes + (size_t)2 * nranks * cap * (sizeof(double) + 16);   // plain inbox + LL cells
        CUDA_CHECK(cudaMalloc(&region, bytes));
        CUDA_CHECK(cudaMemset(region, 0, bytes));
        CUDA_CHECK(cudaDeviceSynchronize());
        LocalGroup& g = local_group(local_group_id);
        std::unique_lock<std::mutex> lk(g.mu);
        if (g.published == 0) { g.nranks = nranks; g.closed = 0; }
        if (g.nranks != nranks || g.region[rank]) throw std::invalid_argument("bioen_b200: inconsistent local group");
        g.region[rank] = region;
        g.device[rank] = device;
        ++g.published;
        g.cv.notify_all();
        if (!g.cv.wait_for(lk, std::chrono::seconds(120), [&] { return g.published == g.nranks; }))
            throw std::runtime_error("bioen_b200: local group did not assemble within 120 s");
        for (int r = 0; r < nranks; ++r) {
            mapped[r] = g.region[r];
            if (g.device[r] != device) {
                cudaError_t e = cudaDeviceEnablePeerAccess(g.device[r], 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CUDA_CHECK(e);
                cudaGetLastError();
            }
        }
        p2p = true;
    }
    // Map every rank's inbox into this process.  Collective: every rank must call it.  Any failure on any rank
    // (no peer access, IPC not permitted in this container, ...) leaves all ranks on the NCCL path.
    void enable_p2p(long long cap_doubles, cudaStream_t st) {
        read_timeout_env();
        const char* env = getenv("BIOEN_B200_P2P");
        int fail = (env && env[0] == '0') || nranks > kP2PMaxRanks;
        cap = cap_doubles;
        const size_t bytes = kP2PHeaderBytes + (size_t)2 * nranks * cap * (sizeof(double) + 16);   // plain inbox + LL cells
        cudaIpcMemHandle_t mine;
        memset(&mine, 0, sizeof(mine));
        if (!fail) {
            if (cudaMalloc(&region, bytes) != cudaSuccess || cudaMemset(region, 0, bytes) != cudaSuccess ||
                cudaDeviceSynchronize() != cudaSuccess || cudaIpcGetMemHandle(&mine, region) != cudaSuccess)
                fail = 1;
        }
        // exchange the 64-byte handles (+ a failure word) through NCCL
        static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t size");
        constexpr int W = 9;  // doubles per rank: 8 handle words + failure flag
        double h_send[W], *d_send = nullptr, *d_all = nullptr;
        std::vector<double> h_all((size_t)W * nranks);
        memcpy(h_send, &mine, 64);
        h_send[8] = fail ? 1.0 : 0.0;
        CUDA_CHECK(cudaMalloc(&d_send, sizeof(h_send)));
        CUDA_CHECK(cudaMalloc(&d_all, h_all.size() * sizeof(double)));
        CUDA_CHECK(cudaMemcpyAsync(d_send, h_send, sizeof(h_send), cudaMemcpyHostToDevice, st));
        nccl_allgather(d_send, d_all, W, st);
        CUDA_CHECK(cudaMemcpyAsync(h_all.data(), d_all, h_all.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        for (int r = 0; r < nranks; ++r) fail |= (h_all[(size_t)r * W + 8] != 0.0);
        if (!fail) {
            for (int r = 0; r < nranks && !fail; ++r) {
                if (r == rank) { mapped[r] = region; continue; }
                cudaIpcMemHandle_t h;
                memcpy(&h, &h_all[(size_t)r * W], 64);
                void* ptr = nullptr;
                if (cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) fail = 1;
                else mapped[r] = static_cast<unsigned char*>(ptr);
            }
        }
        // agree on the outcome; this all-gather is also the barrier behind which every inbox is zeroed and mapped
        h_send[8] = fail ? 1.0 : 0.0;
        CUDA_CHECK(cudaMemcpyAsync(d_send, h_send, sizeof(h_send), cudaMemcpyHostToDevice, st));
        nccl_allgather(d_send, d_all, W, st);
        CUDA_CHECK(cudaMemcpyAsync(h_all.data(), d_all, h_all.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        for (int r = 0; r < nranks; ++r) fail |= (h_all[(size_t)r * W + 8] != 0.0);
        cudaFree(d_send);
        cudaFree(d_all);
        if (fail) {
            release_p2p();
            (void)cudaGetLastError();  // a refused IPC call is not an error of the path: NCCL carries it
        } else {
            p2p = true;
        }
    }
    void release_p2p() {
        if (is_local()) {
            // the table entry is cleared when the last rank of the group leaves (regions of peers may still be in use
            // by their own streams until then; every rank synchronises its stream before destroying its context)
            LocalGroup& g = local_group(local_group_id);
            std::unique_lock<std::mutex> lk(g.mu);
            if (p2p && ++g.closed == g.nranks) {
                g.published = g.closed = g.nranks = 0;
                for (auto& r : g.region) r = nullptr;
            }
            for (auto& m : mapped) m = nullptr;
        }
        for (int r = 0; r < kP2PMaxRanks; ++r) {
            if (mapped[r] && r != rank) cudaIpcCloseMemHandle(mapped[r]);
            mapped[r] = nullptr;
        }
        if (region) cudaFree(region);
        region = nullptr;
        p2p = false;
    }
    // 0: single rank / none, 1: NCCL, 2: peer-memory kernel
    int mode() const { return nranks <= 1 ? 0 : (p2p && use_p2p ? 2 : 1); }
    int exchanges = 0;   // p2p exchanges (separate launches + fused into producers) enqueued so far

    void need_nccl() const {
        if (!comm) throw std::runtime_error("bioen_b200: message too large for the peer-memory inbox and this group "
                                            "has no NCCL communicator (in-process group)");
    }
    void allreduce_sum(double* buf, size_t count, cudaStream_t st) {
        if (exchange(buf, buf, count, kP2PSum, st)) return;
        need_nccl();
        check(NcclApi::get().AllReduce(buf, buf, count, NcclApi::kFloat64, NcclApi::kSum, comm, st), "ncclAllReduce");
    }
    void allreduce_max(double* buf, size_t count, cudaStream_t st) {
        if (exchange(buf, buf, count, kP2PMax, st)) return;
        need_nccl();
        check(NcclApi::get().AllReduce(buf, buf, count, NcclApi::kFloat64, NcclApi::kMax, comm, st), "ncclAllReduce");
    }
    void allgather(const double* send, double* recv, size_t count, cudaStream_t st) {
        if (exchange(send, recv, count, kP2PGather, st)) return;
        nccl_allgather(send, recv, count, st);
    }

   private:
    void nccl_allgather(const double* send, double* recv, size_t count, cudaStream_t st) {
        need_nccl();
        check(NcclApi::get().AllGather(send, recv, count, NcclApi::kFloat64, comm, st), "ncclAllGather");
    }
    bool exchange(const double* send, double* recv, size_t count, int op, cudaStream_t st) {
        if (!(p2p && use_p2p) || count > (size_t)cap) return false;
        NvtxRange nvtx("bioen:p2p_exchange");
        ++exchanges;
        P2PArgs a{};
        a.dev = dev_args();
        a.send = send; a.recv = recv; a.count = (int)count; a.op = op;
        k_p2p_exchange<<<1, kP2PThreads, 0, st>>>(a);
        CUDA_CHECK(cudaGetLastError());
        ++p2p_launches;
        return true;
    }
    static void check(int rc, const char* what) {
        if (rc != 0)
            throw std::runtime_error(std::string("bioen_b200: ") + what + " failed: " +
                                     NcclApi::get().GetErrorString(rc));
    }
};

}  // namespace bioen
