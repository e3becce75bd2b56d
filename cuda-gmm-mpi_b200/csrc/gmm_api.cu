// gmm_api.cu — the C ABI of include/gmm.h: context, operators, EM loop,
// model-order reduction.  Host orchestration in C++, compute in the CUDA
// kernels of kernels_simt.cuh / kernels_tc.cuh, cross-GPU reduction of the
// packed sufficient statistics once per iteration (allreduce_peer_kernel over
// NVLink peer memory, ncclAllReduce where the peers cannot be mapped).
//
// Reference being replaced: gaussian.cu:289-960 (the OpenMP-thread-per-GPU body
// of main()).  There is no CPU fallback: every compute entry point needs a
// CUDA device of compute capability 10.x.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <fcntl.h>
#include <unistd.h>
#include <nccl.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <functional>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <string>
#include <thread>
#include <vector>

#include "../../include/gmm.h"
#include "host_math.h"
#include "kernels_simt.cuh"
#include "kernels_tc.cuh"

namespace gmm {

#define CUDA_TRY(expr)                                                                        \
    do {                                                                                      \
        cudaError_t e_ = (expr);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return fail(GMM_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));    \
    } while (0)

// ---- NCCL, loaded lazily so that the library imports without it -----------
struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};
static NcclApi& nccl() {
    static NcclApi api;
    static bool tried = false;
    if (!tried) {
        tried = true;
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* nm : names) {
            api.handle = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
            if (api.handle) break;
        }
        if (api.handle) {
            api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(api.handle, "ncclGetUniqueId");
            api.CommInitRank = (decltype(api.CommInitRank))dlsym(api.handle, "ncclCommInitRank");
            api.AllReduce = (decltype(api.AllReduce))dlsym(api.handle, "ncclAllReduce");
            api.AllGather = (decltype(api.AllGather))dlsym(api.handle, "ncclAllGather");
            api.CommDestroy = (decltype(api.CommDestroy))dlsym(api.handle, "ncclCommDestroy");
            api.GetErrorString = (decltype(api.GetErrorString))dlsym(api.handle, "ncclGetErrorString");
            api.ok = api.GetUniqueId && api.CommInitRank && api.AllReduce && api.AllGather && api.CommDestroy && api.GetErrorString;
        }
    }
    return api;
}
#define NCCL_TRY(expr)                                                                         \
    do {                                                                                       \
        ncclResult_t r_ = (expr);                                                              \
        if (r_ != ncclSuccess)                                                                 \
            return fail(GMM_ERR_NCCL, std::string(#expr) + ": " + nccl().GetErrorString(r_));  \
    } while (0)

struct PhaseTimer {          // replaces cudaTimer_t / profile_t (gaussian.cu:33-106)
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending;
    double total_ms = 0;
};
// Timing events are recycled: cudaEventCreate / Destroy cost microseconds each and sat inside the EM loop.
struct EventPool {
    std::vector<cudaEvent_t> free_list;
    cudaEvent_t get() {
        if (!free_list.empty()) { cudaEvent_t e = free_list.back(); free_list.pop_back(); return e; }
        cudaEvent_t e = nullptr;
        cudaEventCreate(&e);
        return e;
    }
    void put(cudaEvent_t e) { if (e) free_list.push_back(e); }
    void destroy() { for (cudaEvent_t e : free_list) cudaEventDestroy(e); free_list.clear(); }
};

// ---------------------------------------------------------------------------------------------------------------
// All-reduce of the packed statistics over NVLink peer memory (one box, <= 8 GPUs): replaces the per-iteration
// ncclAllReduce (and with it the four MPI_Allreduce of gaussian.cu:566,605,658,741) by ONE kernel of this library.
// Every rank owns an exchange area [2 parities][len doubles] + flags, mapped into every other rank (cudaIpc between
// processes, peer access between the threads of one process; NCCL only carries the 100-byte handles once, at
// gmm_comm_init).  Per call and CTA: copy the CTA's chunk of the local statistics into the own area, fence, raise
// the chunk's flag in every peer (posted remote writes), wait for the G flags of the chunk in LOCAL memory, then sum
// the chunk over the ranks' areas in rank order (remote loads) — the same order on every rank, so the replicated host
// finalisation sees bit-identical statistics.  Two parities: a rank can be at most one call ahead of the slowest one.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kXMaxRanks = 8;
constexpr int kXCtas = 24;                      // chunks of the vector, one CTA each (flags per chunk: no grid barrier)
struct PeerTable {
    double* buf[kXMaxRanks];                    // exchange area of rank p as mapped HERE: [2][cap] doubles
    unsigned long long* flags[kXMaxRanks];      // flags of rank p as mapped here: [2][kXMaxRanks][kXCtas]
    int nranks, rank;
    size_t cap;
};
struct PeerExchange {
    PeerTable tab{};
    void* base = nullptr;                       // own allocation: [2][cap] doubles, then the flags
    void* opened[kXMaxRanks] = {nullptr};       // cudaIpcOpenMemHandle results to close
    unsigned long long epoch = 0;
    bool ok = false;
};
struct PeerHello {                              // what every rank tells the others (carried by ncclAllGather once)
    cudaIpcMemHandle_t handle;
    unsigned long long ptr;
    long long pid;
    int device, ok;
    int dev_fin, pad;                           // this rank can finalise on the device (it has events and the buffers)
};

__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ double ld_relaxed_sys(const double* p) {
    double v;
    asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}

__global__ void __launch_bounds__(1024)
allreduce_peer_kernel(PeerTable t, double* __restrict__ stats, int len, int parity, unsigned long long epoch) {
    const int per = (len + kXCtas - 1) / kXCtas;
    const int i0 = blockIdx.x * per, i1 = min(len, i0 + per);
    double* mine = t.buf[t.rank] + (size_t)parity * t.cap;
    for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) mine[i] = stats[i];
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x < t.nranks)                  // tell rank threadIdx.x that this chunk of rank t.rank is in place
        st_release_sys(t.flags[threadIdx.x] + ((size_t)parity * kXMaxRanks + t.rank) * kXCtas + blockIdx.x, epoch);
    __shared__ int timed_out;
    if (threadIdx.x == 0) timed_out = 0;
    __syncthreads();
    if (threadIdx.x < t.nranks) {
        const unsigned long long* f = t.flags[t.rank] + ((size_t)parity * kXMaxRanks + threadIdx.x) * kXCtas + blockIdx.x;
        const long long t0 = clock64();
        while (ld_acquire_sys(f) < epoch) {
            __nanosleep(20);
            if (clock64() - t0 > 20000000000LL) { timed_out = 1; break; }      // ~10 s: a peer is gone; do not hang the GPU
        }
    }
    __syncthreads();
    for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
        double s = 0.0;
        for (int p = 0; p < t.nranks; p++) s += ld_relaxed_sys(t.buf[p] + (size_t)parity * t.cap + i);
        stats[i] = timed_out ? __longlong_as_double(0x7ff8000000000000LL) : s;   // NaN: the host reports the failure
    }
}

}  // namespace gmm

using namespace gmm;

struct gmm_ctx {
    int device = 0, n = 0, D = 0, Kmax = 0, F = 0;
    long long n_global = 0, offset = 0;
    cudaStream_t stream = nullptr;
    int num_sms = 148;
    // events
    float* d_x_aos = nullptr;    // [n][D]  as supplied (TMA source of the tensor path)
    float* d_x_soa = nullptr;    // [D][n]  transpose for the SIMT kernels
    // responsibilities, cluster-major [Kmax][n]
    float* d_memb = nullptr;
    size_t memb_pitch = 0;           // row pitch in floats (multiple of 32: TMA-aligned rows)
    float* d_memb_saved = nullptr;   // best configuration during gmm_fit
    cudaEvent_t ev_stats = nullptr;  // statistics have reached the host
    // parameters
    float* d_epack = nullptr;    // SIMT E-step parameters [Kmax][epack_stride]
    float* h_epack = nullptr;    // pinned staging
    double* d_stats = nullptr;   // [Kmax*F + 1]
    double* h_stats = nullptr;   // pinned
    double* d_shift = nullptr;   // [32]
    double shift[GMM_MAX_DIMENSIONS] = {0};
    bool have_shift = false;
    double scale[GMM_MAX_DIMENSIONS] = {0};   // global per-dimension standard deviation
    double sum_x[GMM_MAX_DIMENSIONS] = {0}, sum_x2[GMM_MAX_DIMENSIONS] = {0};
    // host copy of the current parameters (all arrays sized for Kmax)
    std::vector<float> hN, hpi, hconst, havgvar, hmeans, hR, hRinv;
    clusters_t host{};
    int cur_K = 0;
    bool memb_valid = false;     // d_memb holds the responsibilities of the current parameters
    int stats_clean_K = 0;       // d_stats[0 .. K*F) is known to be zero for this K (0 = not known)
    // communication
    ncclComm_t comm = nullptr;
    int rank = 0, nranks = 1;
    // options
    int path = GMM_PATH_AUTO;
    int estep_path = -1, mstep_path = -1;   // per-step override of `path` (options "estep_path" / "mstep_path"; -1 = follow `path`)
    int verbose = 0;
    int host_threads = 1;
    bool host_threads_fixed = false; // set by GMM_HOST_THREADS / gmm_set_option: not re-derived from the rank count
    // profile
    PhaseTimer t_estep, t_mstep, t_reduce;
    EventPool events;
    bool profile_phases = true;  // per-phase CUDA-event timers inside the EM loop (option "profile")
    double host_const_ms = 0, memcpy_ms = 0;
    double fit_reduce_ms = 0, fit_seed_ms = 0, fit_save_ms = 0;   // gmm_fit phases (gmm_get_fit_profile)
    long long mstep_tensor = 0, mstep_simt = 0;                   // M-step launches by kernel
    long long iterations = 0;
    TcState* tc = nullptr;       // tensor-core path state (kernels_tc.cuh)
    HostPool pool{1};            // worker team of the host's loops over clusters (host_pool() sizes it)
    PeerExchange xchg;           // peer-memory all-reduce of the statistics (gmm_comm_init; falls back to NCCL)
    int allreduce_mode = 1;      // option "allreduce": 1 = peer-memory kernel when available, 0 = ncclAllReduce
    bool estep_tensor_ready = false;   // the tensor E-step operand of the current parameters is uploaded
    // device-side finalisation (kernels_tc.cu: finalize_params_kernel): EM iterations without a host round trip
    int finalize_mode = 1;       // option "finalize": 1 = on the device when the tensor E-step serves the state, 0 = host
    bool dev_fin_failed = false; // a cluster needed the host path once: this context stays on it
    bool dev_fin_agreed = true;  // every rank of the communicator can (gmm_comm_init): the replay re-issues collectives
    float* d_pset[2] = {nullptr, nullptr};   // parameter sets written by the kernel (iteration parity)
    float* h_pset = nullptr;     // pinned staging of one set
    float* d_avgvar = nullptr;   // [Kmax]
    int* d_bad = nullptr;        // [2] first failed iteration (-1), code
    double* d_llprev = nullptr;  // [2] log-likelihood slot seen by the finalisation of iteration parity
    struct DevFinStaging {       // pinned staging of the small transfers around the device-side finalisation
        int bad_in[2];           // -> d_bad before a batch: no failure yet
        int bad_out[2];          // <- d_bad after it
        double ll[2];            // <- d_llprev
        float avgvar[GMM_MAX_CLUSTERS];   // -> d_avgvar when the parameters are set from outside
    }* h_fin = nullptr;
    PhaseTimer t_final;
    long long dev_finalize_launches = 0, dev_replays = 0;
    int fin_fault_iter = -1;     // option "finalize_fault_iter" (tests): that iteration of the next batch reports a failure
};

namespace gmm {

static void timer_begin(gmm_ctx* c, PhaseTimer& t) {
    if (!c->profile_phases) return;
    cudaEvent_t a = c->events.get(), b = c->events.get();
    cudaEventRecord(a, c->stream);
    t.pending.push_back({a, b});
}
static void timer_end(gmm_ctx* c, PhaseTimer& t) {
    if (!c->profile_phases || t.pending.empty()) return;
    cudaEventRecord(t.pending.back().second, c->stream);
}
static void timer_collect(gmm_ctx* c, PhaseTimer& t) {          // call after a stream sync
    for (auto& p : t.pending) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, p.first, p.second) == cudaSuccess) t.total_ms += ms;
        c->events.put(p.first); c->events.put(p.second);
    }
    t.pending.clear();
}
static void collect_all(gmm_ctx* c) {
    timer_collect(c, c->t_estep); timer_collect(c, c->t_mstep); timer_collect(c, c->t_reduce); timer_collect(c, c->t_final);
}

static void bind_host(gmm_ctx* c) {
    c->host.N = c->hN.data(); c->host.pi = c->hpi.data(); c->host.constant = c->hconst.data();
    c->host.avgvar = c->havgvar.data(); c->host.means = c->hmeans.data(); c->host.R = c->hR.data();
    c->host.Rinv = c->hRinv.data(); c->host.memberships = nullptr;
}

static void copy_params(clusters_t* dst, const clusters_t* src, int K, int D) {
    std::memcpy(dst->N, src->N, sizeof(float) * K);
    std::memcpy(dst->pi, src->pi, sizeof(float) * K);
    std::memcpy(dst->constant, src->constant, sizeof(float) * K);
    std::memcpy(dst->avgvar, src->avgvar, sizeof(float) * K);
    std::memcpy(dst->means, src->means, sizeof(float) * (size_t)K * D);
    std::memcpy(dst->R, src->R, sizeof(float) * (size_t)K * D * D);
    std::memcpy(dst->Rinv, src->Rinv, sizeof(float) * (size_t)K * D * D);
}

// Threads of the replicated host finalisation (K independent D x D inversions + factorizations, ~5 us each): at most
// 16 (beyond that the fork/join costs more than it saves) and at most HALF of this rank's share of the hardware
// threads — with every hardware thread of the box claimed by spinning thread teams (8 ranks x 16 on 128) the
// NCCL proxy threads starve: measured 3.4 ms per all-reduce and 1.8 ms per finalisation instead of 0.05 / 0.1 ms.
static int default_host_threads(int ranks_on_box) {
    const int hw = (int)std::thread::hardware_concurrency();
    int t = hw > 0 ? hw / (2 * (ranks_on_box > 0 ? ranks_on_box : 1)) : 8;
    if (t > 16) t = 16;
    if (t < 1) t = 1;
    return t;
}

static HostPool& host_pool(gmm_ctx* c) {
    c->pool.resize(c->host_threads);
    return c->pool;
}

static int nccl_allreduce(gmm_ctx* c, double* buf, size_t n, ncclRedOp_t op) {
    const ncclResult_t r = nccl().AllReduce(buf, buf, n, ncclDouble, op, c->comm, c->stream);
    if (r != ncclSuccess) return fail(GMM_ERR_NCCL, std::string("ncclAllReduce: ") + nccl().GetErrorString(r));
    return GMM_OK;
}

static int estep_path_of(const gmm_ctx* c) { return c->estep_path >= 0 ? c->estep_path : c->path; }
static int mstep_path_of(const gmm_ctx* c) { return c->mstep_path >= 0 ? c->mstep_path : c->path; }
static bool use_tensor_estep(const gmm_ctx* c, int K) { return estep_path_of(c) != GMM_PATH_SIMT && c->n > 0 && tc_estep_supported(c->D, K); }
// (the tensor M-step also needs the data range to fit its fixed-point operand budget: known once the moments are)
static bool use_tensor_mstep(const gmm_ctx* c, int K) {
    return mstep_path_of(c) != GMM_PATH_SIMT && c->n > 0 && tc_mstep_supported(c->D, K) && (!c->have_shift || tc_mstep_ready(c->tc));
}
// GMM_PATH_TENSOR never degrades silently: the M-step (the covariance contraction) must be covered.
static int check_path(const gmm_ctx* c, int K) {
    if (mstep_path_of(c) == GMM_PATH_TENSOR && !tc_mstep_supported(c->D, K))
        return fail(GMM_ERR_ARG, "GMM_PATH_TENSOR requested but the tcgen05 kernels do not cover this (D, K)");
    if (mstep_path_of(c) == GMM_PATH_TENSOR && c->n > 0 && c->have_shift && !tc_mstep_ready(c->tc))
        return fail(GMM_ERR_ARG, "GMM_PATH_TENSOR requested but the data range (outliers beyond 64 standard deviations) exceeds the "
                                 "tensor M-step's fixed-point operand budget");
    return GMM_OK;
}

static int ensure_moments(gmm_ctx* c);

// Where the parameters upload_params() sends to the E-step come from: the host copy as given (gmm_seed, gmm_set_clusters,
// gmm_constants, order reduction), or the host finalisation of the reduced statistics in c->h_stats (an EM iteration).
enum class Params { as_given, from_stats };

// Upload the current host parameters in the form the E-step kernels consume (gaussian.cu:446-452 / 935-941 upload the
// seven raw arrays; here the E-step operand is pre-packed on the host once per iteration).  Params::from_stats first
// derives them: N, means, R (gaussian.cu:611-622, 663-679), then inverse + constant (:698-708) from one Cholesky
// factorisation of R (the no-pivot LU where R is not positive definite) and pi.  ONE loop over the clusters on the
// worker team does the per-cluster part of both, and builds the tensor E-step operand when that kernel serves the state.
static int upload_params(gmm_ctx* c, int K, Params src = Params::as_given) {
    if (int rc = check_path(c, K)) return rc;
    auto t0 = std::chrono::steady_clock::now();
    const bool from_stats = src == Params::from_stats;
    const int D = c->D;
    c->estep_tensor_ready = false;
    bool tensor = use_tensor_estep(c, K);
    if (tensor) {
        if (int rc = ensure_moments(c)) return rc;
        // events further than 2^14 global standard deviations from the centre would overflow the FP16 event operand
        const int rc = tc_estep_range_ok(c->tc) ? tc_params_begin(c->tc, K, c->stream)
                                                : fail(GMM_ERR_STATE, "tensor E-step: the data range exceeds the FP16 event operand");
        if (rc != GMM_OK && (rc != GMM_ERR_STATE || estep_path_of(c) == GMM_PATH_TENSOR)) return rc;
        tensor = rc == GMM_OK;
    }
    if (from_stats) {                                      // pi needs every N[k] = (float)S0 before the per-cluster loop
        for (int k = 0; k < K; k++) c->host.N[k] = (float)c->h_stats[(size_t)k * c->F];
        mixing_weights(K, &c->host);
    }
    std::atomic<int> bad_all{0};
    const std::function<void(int)> per_cluster = [&](int k) {
        double W[GMM_MAX_DIMENSIONS * GMM_MAX_DIMENSIONS];
        bool have_w = false;                               // one factorisation serves Rinv, ln det and the operand
        if (from_stats && k < K) {
            finalize_cluster(c->h_stats, c->shift, k, D, &c->host);
            have_w = constants_cluster_spd(k, D, &c->host, W);
            if (!have_w) constants_cluster(k, D, &c->host);
        }
        if (!tensor) return;
        const int b = have_w ? tc_params_cluster_w(c->tc, &c->host, k, K, W) : tc_params_cluster(c->tc, &c->host, k, K);
        int cur = bad_all.load(std::memory_order_relaxed);
        while (b > cur && !bad_all.compare_exchange_weak(cur, b)) {}
    };
    const int n = tensor ? tc_params_padded(c->tc, K) : K;
    if (K >= 8) host_pool(c).run(n, per_cluster);
    else for (int k = 0; k < n; k++) per_cluster(k);
    if (tensor) {
        const int rc = tc_params_commit(c->tc, K, bad_all.load(), c->stream);
        if (rc != GMM_OK && (rc != GMM_ERR_STATE || estep_path_of(c) == GMM_PATH_TENSOR)) return rc;
        // GMM_ERR_STATE under GMM_PATH_AUTO: a cluster whose inverse covariance is not positive definite
        // (or does not fit FP16) — this parameter set is evaluated by the FP32 SIMT kernel instead.
        c->estep_tensor_ready = rc == GMM_OK;
    }
    if (!c->estep_tensor_ready) {
        build_epack(K, D, &c->host, c->h_epack);
        CUDA_TRY(cudaMemcpyAsync(c->d_epack, c->h_epack, sizeof(float) * (size_t)K * epack_stride(D),
                                 cudaMemcpyHostToDevice, c->stream));
    }
    if (c->d_avgvar && c->estep_tensor_ready && !from_stats) {   // the device-side finalisation adds avgvar to the diagonals
        std::memcpy(c->h_fin->avgvar, c->host.avgvar, sizeof(float) * (size_t)K);
        CUDA_TRY(cudaMemcpyAsync(c->d_avgvar, c->h_fin->avgvar, sizeof(float) * (size_t)K, cudaMemcpyHostToDevice, c->stream));
    }
    c->cur_K = K;
    c->memcpy_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return GMM_OK;
}

// ---- kernel dispatch -------------------------------------------------------
template <int D>
static void launch_estep_simt_d(gmm_ctx* c, int K) {
    const int blocks = (c->n + kEstepThreads - 1) / kEstepThreads;
    estep_simt_kernel<D><<<blocks, kEstepThreads, 0, c->stream>>>(c->d_x_soa, c->memb_pitch, c->n, K, c->d_epack, c->d_memb, c->memb_pitch,
                                                                 c->d_stats + (size_t)K * c->F);
}
static int launch_estep_simt(gmm_ctx* c, int K) {
    if (c->n == 0) return GMM_OK;
    switch (c->D) {
#define GMM_CASE(d) case d: launch_estep_simt_d<d>(c, K); break;
        GMM_CASE(1) GMM_CASE(2) GMM_CASE(3) GMM_CASE(4) GMM_CASE(5) GMM_CASE(6) GMM_CASE(7) GMM_CASE(8)
        GMM_CASE(9) GMM_CASE(10) GMM_CASE(11) GMM_CASE(12) GMM_CASE(13) GMM_CASE(14) GMM_CASE(15) GMM_CASE(16)
        GMM_CASE(17) GMM_CASE(18) GMM_CASE(19) GMM_CASE(20) GMM_CASE(21) GMM_CASE(22) GMM_CASE(23) GMM_CASE(24)
        GMM_CASE(25) GMM_CASE(26) GMM_CASE(27) GMM_CASE(28) GMM_CASE(29) GMM_CASE(30) GMM_CASE(31) GMM_CASE(32)
#undef GMM_CASE
        default: return fail(GMM_ERR_ARG, "unsupported dimension count");
    }
    CUDA_TRY(cudaGetLastError());
    return GMM_OK;
}

template <int JMAX, int CPT>
static int launch_mstep_simt_t(gmm_ctx* c, int K) {
    constexpr int FP = 16 * JMAX, KT = 16 * CPT, GS = KT + 2;
    const size_t smem = sizeof(double) * (size_t)(kMstepTE * FP + kMstepTE * GS + kMstepTE * GMM_MAX_DIMENSIONS) +
                        sizeof(short) * 2 * FP;
    // the attribute is per device (context): one flag per device, not per process (a thread per GPU in the CLI)
    static bool attr_set[64] = {false};
    if (c->device >= 64 || !attr_set[c->device]) {
        CUDA_TRY(cudaFuncSetAttribute(mstep_simt_kernel<JMAX, CPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        if (c->device < 64) attr_set[c->device] = true;
    }
    int gx = c->num_sms;
    int per = (c->n + gx - 1) / gx;
    per = (per + kMstepTE - 1) / kMstepTE * kMstepTE;
    if (per < kMstepTE) per = kMstepTE;
    gx = (c->n + per - 1) / per;
    dim3 grid(gx, (K + KT - 1) / KT);
    mstep_simt_kernel<JMAX, CPT><<<grid, kMstepThreads, smem, c->stream>>>(c->d_x_soa, c->memb_pitch, c->n, c->D, K, c->d_memb, c->memb_pitch,
                                                                           c->d_shift, c->d_stats, per);
    CUDA_TRY(cudaGetLastError());
    return GMM_OK;
}
static int launch_mstep_simt(gmm_ctx* c, int K) {
    if (c->n == 0) return GMM_OK;
    const int F = c->F;
    const int cpt = K <= 16 ? 1 : (K <= 32 ? 2 : 4);
    if (F <= 48) {
        if (cpt == 1) return launch_mstep_simt_t<3, 1>(c, K);
        if (cpt == 2) return launch_mstep_simt_t<3, 2>(c, K);
        return launch_mstep_simt_t<3, 4>(c, K);
    } else if (F <= 160) {
        if (cpt == 1) return launch_mstep_simt_t<10, 1>(c, K);
        if (cpt == 2) return launch_mstep_simt_t<10, 2>(c, K);
        return launch_mstep_simt_t<10, 4>(c, K);
    } else if (F <= 336) {
        if (cpt == 1) return launch_mstep_simt_t<21, 1>(c, K);
        if (cpt == 2) return launch_mstep_simt_t<21, 2>(c, K);
        return launch_mstep_simt_t<21, 4>(c, K);
    } else {
        if (cpt == 1) return launch_mstep_simt_t<36, 1>(c, K);
        return launch_mstep_simt_t<36, 2>(c, K);
    }
}

static int zero_stats(gmm_ctx* c, int K) {
    CUDA_TRY(cudaMemsetAsync(c->d_stats, 0, sizeof(double) * ((size_t)K * c->F + 1), c->stream));
    c->stats_clean_K = K;
    return GMM_OK;
}

// E-step on the current device parameters: responsibilities -> d_memb, local
// log-likelihood added to stats[K*F].
static int run_estep(gmm_ctx* c, int K) {
    timer_begin(c, c->t_estep);
    int rc = c->estep_tensor_ready ? tc_launch_estep(c->tc, K, c->d_stats + (size_t)K * c->F, c->stream)
                                   : launch_estep_simt(c, K);
    timer_end(c, c->t_estep);
    c->memb_valid = (rc == GMM_OK);
    return rc;
}

// M-step accumulation of the local statistics into stats[0 .. K*F).
static int run_mstep_accumulate(gmm_ctx* c, int K) {
    // Both M-step kernels ADD into stats[0 .. K*F): whatever an earlier call left there (column moments, seed rows,
    // the reduced statistics of a finished gmm_em / gmm_mstep) has to go; the log-likelihood slot [K*F] stays.
    if (c->stats_clean_K != K) CUDA_TRY(cudaMemsetAsync(c->d_stats, 0, sizeof(double) * (size_t)K * c->F, c->stream));
    c->stats_clean_K = 0;
    timer_begin(c, c->t_mstep);
    int rc;
    if (use_tensor_mstep(c, K)) { rc = tc_launch_mstep(c->tc, K, c->d_stats, c->stream); c->mstep_tensor++; }
    else { rc = launch_mstep_simt(c, K); c->mstep_simt++; }
    timer_end(c, c->t_mstep);
    return rc;
}

// Sum the packed statistics over all ranks (replaces the four MPI_Allreduce of
// gaussian.cu:516,566,605,658,741 and the OpenMP-master sums) and bring them
// to the host.
static int reduce_stats_device(gmm_ctx* c, int K) {
    const size_t len = (size_t)K * c->F + 1;
    timer_begin(c, c->t_reduce);
    if (c->nranks > 1) {
        if (c->xchg.ok && c->allreduce_mode == 1 && len <= c->xchg.tab.cap) {
            c->xchg.epoch++;
            allreduce_peer_kernel<<<kXCtas, 1024, 0, c->stream>>>(c->xchg.tab, c->d_stats, (int)len, (int)(c->xchg.epoch & 1), c->xchg.epoch);
            CUDA_TRY(cudaGetLastError());
        } else if (int rc = nccl_allreduce(c, c->d_stats, len, ncclSum)) {
            return rc;
        }
    }
    timer_end(c, c->t_reduce);
    return GMM_OK;
}
static int reduce_stats_to_host(gmm_ctx* c, int K) {
    const size_t len = (size_t)K * c->F + 1;
    if (int rc = reduce_stats_device(c, K)) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->h_stats, c->d_stats, sizeof(double) * len, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaEventRecord(c->ev_stats, c->stream));
    CUDA_TRY(cudaEventSynchronize(c->ev_stats));
    if (c->nranks > 1 && std::isnan(c->h_stats[0]))
        return fail(GMM_ERR_NCCL, "statistics all-reduce failed (a rank did not arrive, or a cluster's statistics are not finite)");
    return GMM_OK;
}

// Bring only the log-likelihood slot of the last E-step to the host (summed over ranks).
static int reduce_loglik_to_host(gmm_ctx* c, int K, float* out) {
    const size_t ll = (size_t)K * c->F;
    if (c->nranks > 1)
        if (int rc = nccl_allreduce(c, c->d_stats + ll, 1, ncclSum)) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->h_stats + ll, c->d_stats + ll, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (out) *out = (float)c->h_stats[ll];
    return GMM_OK;
}

// Global column moments (sum x, sum x^2 over ALL events of all ranks), computed once per
// context.  They give (a) the seeding mean / average variance (gaussian_kernel.cu:54-102, with
// quirk Q2 fixed: whole data set, double accumulation) and (b) the centre `shift` and per-
// dimension `scale` about which the M-step statistics are accumulated (DESIGN.md).
static int ensure_moments(gmm_ctx* c) {
    if (c->have_shift) return GMM_OK;
    const int D = c->D;
    c->stats_clean_K = 0;
    // d_stats[0..D) sum x, [D..2D) sum x^2, [2D..3D) max x, [3D..4D) max (-x)
    std::vector<double> init(4 * (size_t)D, 0.0);
    for (int d = 0; d < 2 * D; d++) init[2 * D + d] = -std::numeric_limits<double>::max();
    if (4 * (size_t)D > (size_t)c->Kmax * c->F + 1) return fail(GMM_ERR_STATE, "stats buffer too small for the column moments");
    CUDA_TRY(cudaMemcpyAsync(c->d_stats, init.data(), sizeof(double) * 4 * D, cudaMemcpyHostToDevice, c->stream));
    if (c->n > 0) {
        dim3 grid(std::min(4 * c->num_sms, (c->n + 255) / 256), D);
        column_moments_kernel<<<grid, 256, 0, c->stream>>>(c->d_x_soa, c->memb_pitch, c->n, D, c->d_stats);
        CUDA_TRY(cudaGetLastError());
    }
    if (c->nranks > 1) {
        if (int rc = nccl_allreduce(c, c->d_stats, 2 * D, ncclSum)) return rc;
        if (int rc = nccl_allreduce(c, c->d_stats + 2 * D, 2 * D, ncclMax)) return rc;
    }
    CUDA_TRY(cudaMemcpyAsync(c->h_stats, c->d_stats, sizeof(double) * 4 * D, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    double xmin[GMM_MAX_DIMENSIONS], xmax[GMM_MAX_DIMENSIONS];
    for (int d = 0; d < D; d++) {
        c->sum_x[d] = c->h_stats[d];
        c->sum_x2[d] = c->h_stats[D + d];
        xmax[d] = c->h_stats[2 * D + d];
        xmin[d] = -c->h_stats[3 * D + d];
        const double mean = c->sum_x[d] / (double)c->n_global;
        const double var = c->sum_x2[d] / (double)c->n_global - mean * mean;
        c->shift[d] = mean;
        c->scale[d] = var > 0 ? std::sqrt(var) : 1.0;
    }
    if (int rc = tc_set_shift_scale(c->tc, c->shift, c->scale, xmin, xmax, c->stream)) return rc;   // rounds shift to float in place
    CUDA_TRY(cudaMemcpyAsync(c->d_shift, c->shift, sizeof(double) * D, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    c->have_shift = true;
    return GMM_OK;
}

static int check_K(const gmm_ctx* c, int K, const char* who) {
    if (!c) return fail(GMM_ERR_ARG, std::string(who) + ": null context");
    if (K < 1 || K > c->Kmax) return fail(GMM_ERR_ARG, std::string(who) + ": K out of range");
    return GMM_OK;
}

// The shard's events in d_x_aos (copied from host_aos first unless it is null) -> their SoA transpose for the SIMT kernels.
static int upload_events(gmm_ctx* c, const float* host_aos) {
    if (c->n == 0) return GMM_OK;
    if (host_aos)
        CUDA_TRY(cudaMemcpyAsync(c->d_x_aos, host_aos, sizeof(float) * (size_t)c->n * c->D, cudaMemcpyHostToDevice, c->stream));
    transpose_aos_to_soa_kernel<<<(c->n + 31) / 32, dim3(32, 8), 0, c->stream>>>(c->d_x_aos, c->d_x_soa, c->memb_pitch, c->n, c->D);
    CUDA_TRY(cudaGetLastError());
    return GMM_OK;
}

// After new events: the global moments (shift / scale, seeding statistics) are recomputed on the next collective call,
// and the resident E-step operand was built in the coordinates of the previous data set: the caller has to set
// parameters again (gmm_seed / gmm_set_clusters) before the next E-step.
static void events_replaced(gmm_ctx* c) {
    c->have_shift = false;
    c->memb_valid = false;
    c->estep_tensor_ready = false;
    c->cur_K = 0;
}

}  // namespace gmm

// ===========================================================================
extern "C" {

static int peer_exchange_setup(gmm_ctx* c);
static void peer_exchange_destroy(gmm_ctx* c);

const char* gmm_version(void) { return "cuda-gmm-mpi_b200 0.1 (sm_100a)"; }

int gmm_create(gmm_ctx** out, int device, int n_local, int D, int Kmax, const float* events_aos,
               long long n_global, long long offset) {
    if (!out) return fail(GMM_ERR_ARG, "gmm_create: null out");
    *out = nullptr;
    if (D < 1 || D > GMM_MAX_DIMENSIONS) return fail(GMM_ERR_ARG, "gmm_create: D must be in [1,32] (gaussian.h:16)");
    if (Kmax < 1 || Kmax > GMM_MAX_CLUSTERS) return fail(GMM_ERR_ARG, "gmm_create: Kmax must be in [1,512] (gaussian.h:10)");
    if (n_local < 0) return fail(GMM_ERR_ARG, "gmm_create: bad events");   // events_aos == NULL: supplied later (gmm_upload_events*)
    if (n_global <= 0) n_global = n_local;
    if (n_global < 1) return fail(GMM_ERR_ARG, "gmm_create: no events");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
        return fail(GMM_ERR_CUDA, "ERROR: No CUDA capable GPUs detected (this engine has no CPU fallback).");
    if (device < 0 || device >= ndev) return fail(GMM_ERR_ARG, "gmm_create: device index out of range");
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(GMM_ERR_CUDA, std::string("device '") + prop.name + "' is not sm_100 (B200); kernels are built for sm_100a only");

    gmm_ctx* c = new gmm_ctx();
    c->device = device; c->n = n_local; c->D = D; c->Kmax = Kmax; c->F = num_features(D);
    c->n_global = n_global; c->offset = offset; c->num_sms = prop.multiProcessorCount;
    const char* ht = getenv("GMM_HOST_THREADS");
    c->host_threads_fixed = ht != nullptr;
    c->host_threads = ht ? atoi(ht) : default_host_threads(1);
    if (c->host_threads < 1) c->host_threads = 1;
    c->hN.assign(Kmax, 0); c->hpi.assign(Kmax, 0); c->hconst.assign(Kmax, 0); c->havgvar.assign(Kmax, 0);
    c->hmeans.assign((size_t)Kmax * D, 0); c->hR.assign((size_t)Kmax * D * D, 0); c->hRinv.assign((size_t)Kmax * D * D, 0);
    bind_host(c);
#define CREATE_TRY(expr)                                                                             \
    do {                                                                                             \
        cudaError_t e_ = (expr);                                                                     \
        if (e_ != cudaSuccess) {                                                                     \
            int rc_ = fail(GMM_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));        \
            gmm_destroy(c);                                                                          \
            return rc_;                                                                              \
        }                                                                                            \
    } while (0)
    CREATE_TRY(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CREATE_TRY(cudaEventCreateWithFlags(&c->ev_stats, cudaEventDisableTiming));
    const size_t nmax = n_local > 0 ? (size_t)n_local : 1;
    CREATE_TRY(cudaMalloc(&c->d_x_aos, sizeof(float) * nmax * D));
    c->memb_pitch = (nmax + 31) / 32 * 32;         // also the row pitch of the SoA event copy
    CREATE_TRY(cudaMalloc(&c->d_x_soa, sizeof(float) * c->memb_pitch * D));
    // rows in multiples of 8: the tensor E-step stores whole 8-cluster groups (zeros for the padding clusters)
    CREATE_TRY(cudaMalloc(&c->d_memb, sizeof(float) * c->memb_pitch * (size_t)((Kmax + 7) / 8 * 8)));
    CREATE_TRY(cudaMalloc(&c->d_epack, sizeof(float) * (size_t)Kmax * epack_stride(D)));
    CREATE_TRY(cudaMallocHost(&c->h_epack, sizeof(float) * (size_t)Kmax * epack_stride(D)));
    CREATE_TRY(cudaMalloc(&c->d_stats, sizeof(double) * ((size_t)Kmax * c->F + 1)));
    CREATE_TRY(cudaMemsetAsync(c->d_stats, 0, sizeof(double) * ((size_t)Kmax * c->F + 1), c->stream));
    CREATE_TRY(cudaMallocHost(&c->h_stats, sizeof(double) * ((size_t)Kmax * c->F + 1)));
    CREATE_TRY(cudaMalloc(&c->d_shift, sizeof(double) * GMM_MAX_DIMENSIONS));
    CREATE_TRY(cudaMemsetAsync(c->d_shift, 0, sizeof(double) * GMM_MAX_DIMENSIONS, c->stream));
    if (events_aos)
        if (int rc = upload_events(c, events_aos)) { gmm_destroy(c); return rc; }
    if (int rc = tc_create(&c->tc, c->d_x_aos, c->d_x_soa, n_local, D, Kmax, c->d_memb, c->memb_pitch, c->num_sms, c->stream)) {
        gmm_destroy(c);
        return rc;
    }
    if (const char* fm = getenv("GMM_FINALIZE")) c->finalize_mode = (std::string(fm) == "host") ? 0 : 1;
    if (n_local > 0 && tc_estep_supported(D, Kmax)) {
        const size_t setf = tc_param_set_floats(Kmax, D);
        for (int b = 0; b < 2; b++) CREATE_TRY(cudaMalloc(&c->d_pset[b], sizeof(float) * setf));
        CREATE_TRY(cudaMallocHost(&c->h_pset, sizeof(float) * setf));
        CREATE_TRY(cudaMalloc(&c->d_avgvar, sizeof(float) * (size_t)Kmax));
        CREATE_TRY(cudaMemsetAsync(c->d_avgvar, 0, sizeof(float) * (size_t)Kmax, c->stream));
        CREATE_TRY(cudaMalloc(&c->d_bad, 2 * sizeof(int)));
        CREATE_TRY(cudaMalloc(&c->d_llprev, 2 * sizeof(double)));
        CREATE_TRY(cudaMallocHost(&c->h_fin, sizeof(*c->h_fin)));
    }
    CREATE_TRY(cudaStreamSynchronize(c->stream));
#undef CREATE_TRY
    *out = c;
    return GMM_OK;
}

// Replace the events of this shard (same n_local, D): H2D copy + device transpose.  The global
// moments (shift / scale, seeding statistics) are recomputed on the next collective call.
int gmm_upload_events(gmm_ctx* c, const float* events_aos) {
    if (!c || (c->n > 0 && !events_aos)) return fail(GMM_ERR_ARG, "gmm_upload_events: bad argument");
    CUDA_TRY(cudaSetDevice(c->device));
    if (int rc = upload_events(c, events_aos)) return rc;
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    events_replaced(c);
    return GMM_OK;
}

// The shard's rows of a "*.bin" file (readData.cpp:35-47 format) straight to the device: pread into two pinned
// staging buffers, each chunk's H2D copy overlapping the read of the next (replaces whole-file malloc + fread on the
// host, gaussian.cu:188-218, followed by a pageable copy per GPU, :360-377).
int gmm_upload_events_file(gmm_ctx* c, const char* path) {
    if (!c || !path) return fail(GMM_ERR_ARG, "gmm_upload_events_file: bad argument");
    CUDA_TRY(cudaSetDevice(c->device));
    const int fd = open(path, O_RDONLY);
    if (fd < 0) return fail(GMM_ERR_IO, std::string("cannot open ") + path);
    int32_t hdr[2] = {0, 0};
    if (pread(fd, hdr, sizeof(hdr), 0) != (ssize_t)sizeof(hdr) || hdr[0] <= 0 || hdr[1] != c->D || (long long)hdr[0] != c->n_global) {
        close(fd);
        return fail(GMM_ERR_IO, "gmm_upload_events_file: header does not match the context (events / dimensions)");
    }
    const size_t row = sizeof(float) * (size_t)c->D;
    const size_t total = row * (size_t)c->n;
    const size_t chunk = std::max<size_t>(row, ((size_t)32 << 20) / row * row);
    char* stage[2] = {nullptr, nullptr};
    cudaEvent_t done[2] = {nullptr, nullptr};
    int rc = GMM_OK;
    for (int b = 0; b < 2 && rc == GMM_OK; b++) {
        if (cudaMallocHost(&stage[b], chunk) != cudaSuccess || cudaEventCreateWithFlags(&done[b], cudaEventDisableTiming) != cudaSuccess)
            rc = fail(GMM_ERR_CUDA, "gmm_upload_events_file: pinned staging allocation failed");
    }
    size_t off = 0;
    for (int i = 0; rc == GMM_OK && off < total; i++) {
        const int b = i & 1;
        const size_t len = std::min(chunk, total - off);
        if (i >= 2 && cudaEventSynchronize(done[b]) != cudaSuccess) { rc = fail(GMM_ERR_CUDA, "gmm_upload_events_file: copy failed"); break; }
        size_t got = 0;
        while (got < len) {
            const ssize_t r = pread(fd, stage[b] + got, len - got, (off_t)(sizeof(hdr) + row * (size_t)c->offset + off + got));
            if (r <= 0) { rc = fail(GMM_ERR_IO, "truncated .bin file"); break; }
            got += (size_t)r;
        }
        if (rc != GMM_OK) break;
        if (cudaMemcpyAsync(reinterpret_cast<char*>(c->d_x_aos) + off, stage[b], len, cudaMemcpyHostToDevice, c->stream) != cudaSuccess ||
            cudaEventRecord(done[b], c->stream) != cudaSuccess) { rc = fail(GMM_ERR_CUDA, "gmm_upload_events_file: copy failed"); break; }
        off += len;
    }
    close(fd);
    if (rc == GMM_OK) rc = upload_events(c, nullptr);
    if (cudaStreamSynchronize(c->stream) != cudaSuccess && rc == GMM_OK) rc = fail(GMM_ERR_CUDA, "gmm_upload_events_file: copy failed");
    for (int b = 0; b < 2; b++) {
        if (stage[b]) cudaFreeHost(stage[b]);
        if (done[b]) cudaEventDestroy(done[b]);
    }
    events_replaced(c);
    return rc;
}

void gmm_destroy(gmm_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    collect_all(c);
    peer_exchange_destroy(c);
    if (c->comm && nccl().ok) nccl().CommDestroy(c->comm);
    tc_destroy(c->tc);
    cudaFree(c->d_x_aos); cudaFree(c->d_x_soa); cudaFree(c->d_memb); cudaFree(c->d_memb_saved);
    cudaFree(c->d_epack); cudaFree(c->d_stats); cudaFree(c->d_shift);
    cudaFree(c->d_pset[0]); cudaFree(c->d_pset[1]); cudaFree(c->d_avgvar); cudaFree(c->d_bad); cudaFree(c->d_llprev);
    if (c->h_pset) cudaFreeHost(c->h_pset);
    if (c->h_fin) cudaFreeHost(c->h_fin);
    if (c->h_epack) cudaFreeHost(c->h_epack);
    if (c->h_stats) cudaFreeHost(c->h_stats);
    if (c->ev_stats) cudaEventDestroy(c->ev_stats);
    c->events.destroy();
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

// Maps every rank's exchange area into this rank (see allreduce_peer_kernel).  Never fatal: whatever goes wrong on
// any rank (no peer access, IPC refused, more than 8 ranks) leaves ALL ranks on ncclAllReduce — the decision is itself
// agreed through the gathered `ok` fields.
static int peer_exchange_setup(gmm_ctx* c) {
    PeerExchange& x = c->xchg;
    x.ok = false;
    const int G = c->nranks;
    const size_t cap = (size_t)c->Kmax * c->F + 1;
    const size_t flag_count = (size_t)2 * kXMaxRanks * kXCtas;
    const size_t bytes = sizeof(double) * 2 * cap + sizeof(unsigned long long) * flag_count;
    PeerHello me{};
    me.pid = (long long)getpid();
    me.device = c->device;
    me.ok = G <= kXMaxRanks ? 1 : 0;
    me.dev_fin = c->d_pset[0] ? 1 : 0;
    if (me.ok && cudaMalloc(&x.base, bytes) != cudaSuccess) { x.base = nullptr; me.ok = 0; cudaGetLastError(); }
    if (me.ok) {
        cudaMemset(x.base, 0, bytes);
        me.ptr = (unsigned long long)(uintptr_t)x.base;
        if (cudaIpcGetMemHandle(&me.handle, x.base) != cudaSuccess) { me.ok = 0; cudaGetLastError(); }
    }
    // gather the hellos (device staging; NCCL is the only channel the C ABI has between ranks)
    PeerHello* d_all = nullptr;
    std::vector<PeerHello> all((size_t)G);
    CUDA_TRY(cudaMalloc(&d_all, sizeof(PeerHello) * G));
    CUDA_TRY(cudaMemcpyAsync(d_all + c->rank, &me, sizeof(PeerHello), cudaMemcpyHostToDevice, c->stream));
    {
        ncclResult_t r = nccl().AllGather(d_all + c->rank, d_all, sizeof(PeerHello), ncclChar, c->comm, c->stream);
        if (r != ncclSuccess) { cudaFree(d_all); return fail(GMM_ERR_NCCL, std::string("ncclAllGather: ") + nccl().GetErrorString(r)); }
    }
    CUDA_TRY(cudaMemcpyAsync(all.data(), d_all, sizeof(PeerHello) * G, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    cudaFree(d_all);
    int ok = 1;
    for (int p = 0; p < G; p++) ok &= all[p].ok;
    c->dev_fin_agreed = true;
    for (int p = 0; p < G; p++) c->dev_fin_agreed = c->dev_fin_agreed && all[p].dev_fin != 0;
    x.tab.nranks = G; x.tab.rank = c->rank; x.tab.cap = cap;
    for (int p = 0; p < G && ok; p++) {
        void* mapped = nullptr;
        if (p == c->rank) mapped = x.base;
        else if (all[p].pid == me.pid) {                 // a thread of this process: plain peer access
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, c->device, all[p].device) != cudaSuccess || !can) ok = 0;
            else {
                cudaError_t e = cudaDeviceEnablePeerAccess(all[p].device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) ok = 0;
                cudaGetLastError();
                mapped = (void*)(uintptr_t)all[p].ptr;
            }
        } else {
            if (cudaIpcOpenMemHandle(&mapped, all[p].handle, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { ok = 0; cudaGetLastError(); }
            else x.opened[p] = mapped;
        }
        if (ok) {
            x.tab.buf[p] = reinterpret_cast<double*>(mapped);
            x.tab.flags[p] = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(mapped) + sizeof(double) * 2 * cap);
        }
    }
    // a rank that failed to map somebody must take everybody back to NCCL: agree on the minimum
    {
        double* d_ok = nullptr;
        double h_ok = ok ? 1.0 : 0.0;
        CUDA_TRY(cudaMalloc(&d_ok, sizeof(double)));
        CUDA_TRY(cudaMemcpyAsync(d_ok, &h_ok, sizeof(double), cudaMemcpyHostToDevice, c->stream));
        if (int rc = nccl_allreduce(c, d_ok, 1, ncclMin)) { cudaFree(d_ok); return rc; }
        CUDA_TRY(cudaMemcpyAsync(&h_ok, d_ok, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));
        cudaFree(d_ok);
        ok = h_ok > 0.5;
    }
    x.ok = ok != 0;
    if (c->verbose) std::printf("[gmm rank %d] statistics all-reduce: %s\n", c->rank, x.ok ? "peer-memory kernel (NVLink)" : "ncclAllReduce");
    return GMM_OK;
}

static void peer_exchange_destroy(gmm_ctx* c) {
    PeerExchange& x = c->xchg;
    for (int p = 0; p < kXMaxRanks; p++)
        if (x.opened[p]) { cudaIpcCloseMemHandle(x.opened[p]); x.opened[p] = nullptr; }
    if (x.base) { cudaFree(x.base); x.base = nullptr; }
    x.ok = false;
}

int gmm_nccl_unique_id(char id_out[128]) {
    if (!id_out) return fail(GMM_ERR_ARG, "gmm_nccl_unique_id: null");
    if (!nccl().ok) return fail(GMM_ERR_NCCL, "libnccl.so.2 not found");
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
    ncclUniqueId id;
    NCCL_TRY(nccl().GetUniqueId(&id));
    std::memcpy(id_out, &id, 128);
    return GMM_OK;
}

int gmm_comm_init(gmm_ctx* c, int nranks, int rank, const char id_in[128]) {
    if (!c || nranks < 1 || rank < 0 || rank >= nranks) return fail(GMM_ERR_ARG, "gmm_comm_init: bad argument");
    c->rank = rank; c->nranks = nranks;
    if (!c->host_threads_fixed) c->host_threads = default_host_threads(nranks);   // the ranks of one box share its cores
    if (nranks == 1) return GMM_OK;
    if (!id_in) return fail(GMM_ERR_ARG, "gmm_comm_init: null id");
    if (!nccl().ok) return fail(GMM_ERR_NCCL, "libnccl.so.2 not found");
    CUDA_TRY(cudaSetDevice(c->device));
    ncclUniqueId id;
    std::memcpy(&id, id_in, 128);
    NCCL_TRY(nccl().CommInitRank(&c->comm, nranks, id, rank));
    return peer_exchange_setup(c);
}

int gmm_comm_rank(const gmm_ctx* c, int* rank, int* nranks) {
    if (!c) return fail(GMM_ERR_ARG, "gmm_comm_rank: null context");
    if (rank) *rank = c->rank;
    if (nranks) *nranks = c->nranks;
    return GMM_OK;
}

int gmm_set_option(gmm_ctx* c, const char* key, double value) {
    if (!c || !key) return fail(GMM_ERR_ARG, "gmm_set_option: bad argument");
    const std::string k(key);
    if (k == "path") {
        const int p = (int)value;
        if (p < GMM_PATH_AUTO || p > GMM_PATH_TENSOR) return fail(GMM_ERR_ARG, "gmm_set_option: bad path");
        c->path = p;
    } else if (k == "verbose") c->verbose = (int)value;
    else if (k == "host_threads") {
        c->host_threads = value < 1 ? 1 : (int)value;
        c->host_threads_fixed = true;
    }
    else if (k == "estep_path" || k == "mstep_path") {
        const int p = (int)value;
        if (p < -1 || p > GMM_PATH_TENSOR) return fail(GMM_ERR_ARG, "gmm_set_option: bad path");
        (k == "estep_path" ? c->estep_path : c->mstep_path) = p;
    }
    else if (k == "profile") c->profile_phases = value != 0;
    else if (k == "allreduce") c->allreduce_mode = value != 0 ? 1 : 0;
    else if (k == "finalize") { c->finalize_mode = value != 0 ? 1 : 0; if (value != 0) c->dev_fin_failed = false; }
    else if (k == "finalize_fault_iter") c->fin_fault_iter = (int)value;
    else return fail(GMM_ERR_ARG, "gmm_set_option: unknown key '" + k + "'");
    return GMM_OK;
}

// --- seeding ---------------------------------------------------------------
int gmm_seed(gmm_ctx* c, int K, clusters_t* host_out) {
    if (int rc = check_K(c, K, "gmm_seed")) return rc;
    CUDA_TRY(cudaSetDevice(c->device));
    if (int rc = ensure_moments(c)) return rc;
    const int D = c->D;
    // seed rows (evenly spaced events, gaussian.cu:110-120): the owning shard contributes, the others add zeros
    const size_t len = (size_t)K * D;
    if (len > (size_t)c->Kmax * c->F + 1) return fail(GMM_ERR_STATE, "gmm_seed: stats buffer too small");
    std::vector<double> rows(len, 0.0);
    std::vector<float> tmp(D);
    for (int k = 0; k < K; k++) {
        const long long g = seed_event_index(k, K, c->n_global);
        if (g >= c->offset && g < c->offset + c->n) {
            CUDA_TRY(cudaMemcpyAsync(tmp.data(), c->d_x_aos + (size_t)(g - c->offset) * D, sizeof(float) * D,
                                     cudaMemcpyDeviceToHost, c->stream));
            CUDA_TRY(cudaStreamSynchronize(c->stream));
            for (int d = 0; d < D; d++) rows[(size_t)k * D + d] = tmp[d];
        }
    }
    if (c->nranks > 1) {
        c->stats_clean_K = 0;
        CUDA_TRY(cudaMemcpyAsync(c->d_stats, rows.data(), sizeof(double) * len, cudaMemcpyHostToDevice, c->stream));
        if (int rc = nccl_allreduce(c, c->d_stats, len, ncclSum)) return rc;
        CUDA_TRY(cudaMemcpyAsync(rows.data(), c->d_stats, sizeof(double) * len, cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));
    }
    std::vector<float> seed_rows(len);
    for (size_t i = 0; i < len; i++) seed_rows[i] = (float)rows[i];
    seed_from_moments(c->sum_x, c->sum_x2, c->n_global, D, K, seed_rows.data(), &c->host);
    if (int rc = upload_params(c, K)) return rc;
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    c->memb_valid = false;
    if (host_out) copy_params(host_out, &c->host, K, D);
    return GMM_OK;
}

int gmm_set_clusters(gmm_ctx* c, int K, const clusters_t* in) {
    if (int rc = check_K(c, K, "gmm_set_clusters")) return rc;
    if (!in) return fail(GMM_ERR_ARG, "gmm_set_clusters: null clusters");
    CUDA_TRY(cudaSetDevice(c->device));
    copy_params(&c->host, in, K, c->D);
    c->memb_valid = false;
    if (int rc = upload_params(c, K)) return rc;
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return GMM_OK;
}

int gmm_get_clusters(gmm_ctx* c, int K, clusters_t* out, int with_memberships) {
    if (int rc = check_K(c, K, "gmm_get_clusters")) return rc;
    if (!out) return fail(GMM_ERR_ARG, "gmm_get_clusters: null clusters");
    CUDA_TRY(cudaSetDevice(c->device));
    copy_params(out, &c->host, K, c->D);
    if (with_memberships) {
        if (!out->memberships) return fail(GMM_ERR_ARG, "gmm_get_clusters: memberships requested but pointer is null");
        if (!c->memb_valid) return fail(GMM_ERR_STATE, "gmm_get_clusters: no E-step has run for the current parameters");
        if (c->n > 0)
            CUDA_TRY(cudaMemcpy2DAsync(out->memberships, sizeof(float) * (size_t)c->n, c->d_memb, sizeof(float) * c->memb_pitch,
                                       sizeof(float) * (size_t)c->n, K, cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));
    }
    return GMM_OK;
}

int gmm_estep(gmm_ctx* c, int K, float* loglik_out) {
    if (int rc = check_K(c, K, "gmm_estep")) return rc;
    if (K != c->cur_K) return fail(GMM_ERR_STATE, "gmm_estep: parameters for this K have not been set");
    CUDA_TRY(cudaSetDevice(c->device));
    const size_t ll = (size_t)K * c->F;
    CUDA_TRY(cudaMemsetAsync(c->d_stats + ll, 0, sizeof(double), c->stream));
    if (int rc = run_estep(c, K)) return rc;
    if (int rc = reduce_loglik_to_host(c, K, loglik_out)) return rc;
    collect_all(c);
    return GMM_OK;
}

int gmm_mstep(gmm_ctx* c, int K) {
    if (int rc = check_K(c, K, "gmm_mstep")) return rc;
    if (!c->memb_valid || K != c->cur_K) return fail(GMM_ERR_STATE, "gmm_mstep: run gmm_estep first");
    CUDA_TRY(cudaSetDevice(c->device));
    if (int rc = ensure_moments(c)) return rc;
    const double ll_keep = c->h_stats[(size_t)K * c->F];
    if (int rc = run_mstep_accumulate(c, K)) return rc;         // zeroes stats[0 .. K*F) first
    if (int rc = reduce_stats_to_host(c, K)) return rc;
    c->h_stats[(size_t)K * c->F] = ll_keep;
    // gmm_mstep stops before constants_kernel: N, means, R only (gaussian.cu:538-687)
    finalize_from_stats(c->h_stats, c->shift, K, c->D, &c->host);
    collect_all(c);
    return GMM_OK;
}

int gmm_constants(gmm_ctx* c, int K) {
    if (int rc = check_K(c, K, "gmm_constants")) return rc;
    CUDA_TRY(cudaSetDevice(c->device));
    auto t0 = std::chrono::steady_clock::now();
    constants_from_R(K, c->D, &c->host, host_pool(c));
    c->host_const_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (int rc = upload_params(c, K)) return rc;
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return GMM_OK;
}

// The two halves of one pass of the loop body of gaussian.cu:532-755 on the device-resident responsibilities.
// First: M-step statistics -> all-reduce -> host.  The log-likelihood of the E-step that produced the
// responsibilities rides in the packed buffer and is returned through *prev_loglik.
static int mstep_to_host(gmm_ctx* c, int K, float* prev_loglik) {
    if (int rc = run_mstep_accumulate(c, K)) return rc;
    if (int rc = reduce_stats_to_host(c, K)) return rc;
    if (prev_loglik) *prev_loglik = (float)c->h_stats[(size_t)K * c->F];
    return GMM_OK;
}
// Second: parameters (finalised from those statistics, or as given) -> upload -> E-step (gaussian.cu:713-714).
static int params_to_estep(gmm_ctx* c, int K, Params src) {
    if (int rc = upload_params(c, K, src)) return rc;
    if (int rc = zero_stats(c, K)) return rc;
    return run_estep(c, K);
}
static int em_iteration(gmm_ctx* c, int K, float* prev_loglik) {
    if (int rc = mstep_to_host(c, K, prev_loglik)) return rc;
    if (int rc = params_to_estep(c, K, Params::from_stats)) return rc;
    c->iterations++;
    return GMM_OK;
}

// ---- EM iterations with the finalisation on the device --------------------------------------------------------
static bool dev_finalize_ok(const gmm_ctx* c, int K) {
    return c->finalize_mode == 1 && !c->dev_fin_failed && c->dev_fin_agreed && c->d_pset[0] && c->n > 0 && c->estep_tensor_ready && K == c->cur_K &&
           use_tensor_estep(c, K) && tc_finalize_supported(c->tc, K);
}

// Parameter set `which` (K-prefixes of its arrays) -> pinned staging; valid after the next stream synchronisation.
static int fetch_param_set(gmm_ctx* c, int K, int which) {
    const int D = c->D, Kmax = c->Kmax;
    const size_t cnt[6] = {(size_t)K, (size_t)K, (size_t)K, (size_t)K * D, (size_t)K * D * D, (size_t)K * D * D};
    for (int a = 0; a < 6; a++) {
        const size_t off = tc_param_set_off(Kmax, D, a);
        CUDA_TRY(cudaMemcpyAsync(c->h_pset + off, c->d_pset[which] + off, sizeof(float) * cnt[a], cudaMemcpyDeviceToHost, c->stream));
    }
    return GMM_OK;
}
static void scatter_param_set(gmm_ctx* c, int K) {
    const int D = c->D, Kmax = c->Kmax;
    float* dst[6] = {c->host.N, c->host.pi, c->host.constant, c->host.means, c->host.R, c->host.Rinv};
    const size_t cnt[6] = {(size_t)K, (size_t)K, (size_t)K, (size_t)K * D, (size_t)K * D * D, (size_t)K * D * D};
    for (int a = 0; a < 6; a++) std::memcpy(dst[a], c->h_pset + tc_param_set_off(Kmax, D, a), sizeof(float) * cnt[a]);
}

// `iters` EM iterations queued back to back: M-step -> all-reduce -> finalize_params_kernel -> E-step, nothing returns to
// the host in between.  Afterwards the host copy of the parameters is refreshed from the last set.  *ll_prev receives the
// log-likelihood slot the LAST finalisation saw (the E-step before the last one; gmm_em's convergence test needs it).
// If a finalisation met a cluster only the host path serves (not positive definite, outside FP16), the work queued after
// it was discarded by the kernels themselves: the host takes the last good set, re-creates the responsibilities that
// iteration started from and runs the remaining iterations through its own path; the context then stays on the host path.
static int run_dev_iterations(gmm_ctx* c, int K, int iters, float* ll_prev) {
    if (iters <= 0) return GMM_OK;
    auto* h = c->h_fin;
    h->bad_in[0] = -1; h->bad_in[1] = 0;
    CUDA_TRY(cudaMemcpyAsync(c->d_bad, h->bad_in, sizeof(h->bad_in), cudaMemcpyHostToDevice, c->stream));
    for (int i = 0; i < iters; i++) {
        if (int rc = run_mstep_accumulate(c, K)) return rc;
        if (int rc = reduce_stats_device(c, K)) return rc;
        timer_begin(c, c->t_final);
        int rc = tc_launch_finalize(c->tc, K, c->d_stats, c->d_avgvar, c->d_pset[i & 1], c->d_llprev + (i & 1), c->d_bad, i, c->fin_fault_iter, c->stream);
        timer_end(c, c->t_final);
        if (rc) return rc;
        c->dev_finalize_launches++;
        if (int rc2 = zero_stats(c, K)) return rc2;
        if (int rc2 = run_estep(c, K)) return rc2;
        c->iterations++;
    }
    CUDA_TRY(cudaMemcpyAsync(h->bad_out, c->d_bad, sizeof(h->bad_out), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(h->ll, c->d_llprev, sizeof(h->ll), cudaMemcpyDeviceToHost, c->stream));
    if (int rc = fetch_param_set(c, K, (iters - 1) & 1)) return rc;
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    const int first_bad = h->bad_out[0], code = h->bad_out[1];
    if (first_bad < 0) {
        scatter_param_set(c, K);
        if (ll_prev) *ll_prev = (float)h->ll[(iters - 1) & 1];
        return GMM_OK;
    }
    if (code == 4) return fail(GMM_ERR_NCCL, "statistics all-reduce failed (a rank did not arrive, or a cluster's statistics are not finite)");
    c->dev_fin_failed = true;
    c->dev_replays++;
    if (c->verbose && c->rank == 0)
        std::printf("[gmm] device-side finalisation met a cluster for the host path at iteration %d (code %d): replaying on the host\n", first_bad, code);
    if (first_bad > 0) {                                   // (first_bad == 0: the host copy is still the state before the batch)
        if (int rc = fetch_param_set(c, K, (first_bad - 1) & 1)) return rc;
        CUDA_TRY(cudaStreamSynchronize(c->stream));
        scatter_param_set(c, K);
    }
    c->iterations -= iters - first_bad;
    if (int rc = params_to_estep(c, K, Params::as_given)) return rc;
    float prev = 0.f;
    for (int i = first_bad; i < iters; i++)
        if (int rc = em_iteration(c, K, &prev)) return rc;
    if (ll_prev) *ll_prev = prev;
    return GMM_OK;
}

int gmm_em_iterations(gmm_ctx* c, int K, int iters, float* loglik_out) {
    if (int rc = check_K(c, K, "gmm_em_iterations")) return rc;
    if (!c->memb_valid || K != c->cur_K) return fail(GMM_ERR_STATE, "gmm_em_iterations: run gmm_estep first");
    CUDA_TRY(cudaSetDevice(c->device));
    if (int rc = ensure_moments(c)) return rc;
    if (dev_finalize_ok(c, K)) {
        if (int rc = run_dev_iterations(c, K, iters, nullptr)) return rc;
    } else {
        for (int i = 0; i < iters; i++)
            if (int rc = em_iteration(c, K, nullptr)) return rc;
    }
    if (int rc = reduce_loglik_to_host(c, K, loglik_out)) return rc;
    collect_all(c);
    return GMM_OK;
}

// The EM loop (gaussian.cu:487-755): initial E-step, then
// while(iters < min_iters || (|change| > epsilon && iters < max_iters)).
// The convergence test needs the log-likelihood of the E-step that just ran;
// it rides in the same packed buffer as the M-step statistics, so when the
// test can still go either way the next M-step accumulation is issued before
// the test (and discarded if the loop ends there).
int gmm_em(gmm_ctx* c, int K, int min_iters, int max_iters, float epsilon, float* loglik_out, int* iters_out) {
    if (int rc = check_K(c, K, "gmm_em")) return rc;
    if (K != c->cur_K) return fail(GMM_ERR_STATE, "gmm_em: parameters for this K have not been set (gmm_seed / gmm_set_clusters)");
    CUDA_TRY(cudaSetDevice(c->device));
    if (int rc = ensure_moments(c)) return rc;
    if (epsilon < 0) epsilon = em_epsilon(c->D, c->n_global);
    if (int rc = zero_stats(c, K)) return rc;
    if (int rc = run_estep(c, K)) return rc;                 // initial E-step, gaussian.cu:487-523
    float likelihood = 0, old_likelihood = 0, change = epsilon * 2;
    int iters = 0;
    if (min_iters > 0 && dev_finalize_ok(c, K)) {
        // the first min_iters iterations run whatever the likelihood does (gaussian.cu:532): no convergence test, so no
        // reason to come back to the host between them
        if (int rc = run_dev_iterations(c, K, min_iters, &old_likelihood)) return rc;
        iters = min_iters;
    }
    for (;;) {
        const bool must_continue = iters < min_iters;
        const bool may_continue = iters < max_iters;
        if (!must_continue && !may_continue) {               // the loop ends whatever the change is
            if (int rc = reduce_loglik_to_host(c, K, &likelihood)) return rc;
            break;
        }
        if (int rc = mstep_to_host(c, K, &likelihood)) return rc;
        if (iters > 0) change = likelihood - old_likelihood;
        if (!(must_continue || (std::fabs(change) > epsilon && may_continue))) break;   // gaussian.cu:532
        old_likelihood = likelihood;
        if (int rc = params_to_estep(c, K, Params::from_stats)) return rc;
        iters++;
        c->iterations++;
        if (c->verbose > 1) std::printf("[gmm rank %d] K=%d iter %d\n", c->rank, K, iters);
    }
    collect_all(c);
    if (loglik_out) *loglik_out = likelihood;
    if (iters_out) *iters_out = iters;
    return GMM_OK;
}

int gmm_get_profile(gmm_ctx* c, double out[8], int reset) {
    if (!c || !out) return fail(GMM_ERR_ARG, "gmm_get_profile: bad argument");
    cudaStreamSynchronize(c->stream);
    collect_all(c);
    out[0] = c->t_estep.total_ms; out[1] = c->t_mstep.total_ms; out[2] = c->host_const_ms;
    out[3] = c->t_reduce.total_ms; out[4] = c->memcpy_ms + c->t_final.total_ms; out[5] = (double)c->mstep_tensor;
    out[6] = (double)c->iterations; out[7] = (double)c->mstep_simt;
    if (reset) {
        c->t_estep.total_ms = c->t_mstep.total_ms = c->t_reduce.total_ms = 0;
        c->host_const_ms = c->memcpy_ms = 0; c->iterations = 0; c->t_final.total_ms = 0;
        c->mstep_tensor = c->mstep_simt = 0;
        c->fit_reduce_ms = c->fit_seed_ms = c->fit_save_ms = 0;
    }
    return GMM_OK;
}

int gmm_get_fit_profile(gmm_ctx* c, double out[4]) {
    if (!c || !out) return fail(GMM_ERR_ARG, "gmm_get_fit_profile: bad argument");
    out[0] = c->fit_reduce_ms; out[1] = c->fit_seed_ms; out[2] = c->fit_save_ms;
    out[3] = (double)c->dev_finalize_launches + 1e-3 * (double)(c->dev_replays > 999 ? 999 : c->dev_replays);
    return GMM_OK;
}

// Model-order reduction loop (gaussian.cu:479-960).
int gmm_fit(gmm_ctx* c, int K0, int target_K, int min_iters, int max_iters, clusters_t* saved, int* ideal_K,
            float* min_rissanen_out) {
    if (int rc = check_K(c, K0, "gmm_fit")) return rc;
    if (target_K < 0 || target_K > K0) return fail(GMM_ERR_ARG, "target_num_clusters must be less than equal to num_clusters");
    if (!saved) return fail(GMM_ERR_ARG, "gmm_fit: null saved clusters");
    CUDA_TRY(cudaSetDevice(c->device));
    const int D = c->D;
    const int stop_number = target_K == 0 ? 1 : target_K;                  // gaussian.cu:177-181
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto ms_since = [](std::chrono::steady_clock::time_point t0) {
        return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    };
    {
        const auto t0 = now();
        if (int rc = gmm_seed(c, K0, nullptr)) return rc;
        c->fit_seed_ms += ms_since(t0);
    }
    const float epsilon = em_epsilon(D, c->n_global);
    float min_rissanen = 0;
    int ideal = K0;
    if (saved->memberships && !c->d_memb_saved && c->n > 0)
        CUDA_TRY(cudaMalloc(&c->d_memb_saved, sizeof(float) * c->memb_pitch * c->Kmax));
    for (int K = K0; K >= stop_number;) {
        float likelihood; int iters;
        if (int rc = gmm_em(c, K, min_iters, max_iters, epsilon, &likelihood, &iters)) return rc;
        const float r = rissanen(likelihood, K, D, c->n_global);          // :826
        if (c->verbose && c->rank == 0) std::printf("K=%d loglik=%e Rissanen Score: %e\n", K, likelihood, r);
        if (K == K0 || (r < min_rissanen && target_K == 0) || K == target_K) {   // :839
            const auto t0 = now();
            min_rissanen = r;
            ideal = K;
            copy_params(saved, &c->host, K, D);
            if (saved->memberships && c->n > 0)
                CUDA_TRY(cudaMemcpyAsync(c->d_memb_saved, c->d_memb, sizeof(float) * (size_t)K * c->memb_pitch, cudaMemcpyDeviceToDevice, c->stream));
            c->fit_save_ms += ms_since(t0);
        }
        if (K > stop_number) {                                            // :860-950
            const auto t0 = now();
            K = reduce_order(&c->host, K, D, nullptr, nullptr, host_pool(c));
            c->fit_reduce_ms += ms_since(t0);
            if (K < 1) break;
            c->memb_valid = false;
            if (int rc = upload_params(c, K)) return rc;
        } else break;
    }
    if (saved->memberships && c->n > 0) {
        CUDA_TRY(cudaMemcpy2DAsync(saved->memberships, sizeof(float) * (size_t)c->n, c->d_memb_saved, sizeof(float) * c->memb_pitch,
                                   sizeof(float) * (size_t)c->n, ideal, cudaMemcpyDeviceToHost, c->stream));
    }
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (ideal_K) *ideal_K = ideal;
    if (min_rissanen_out) *min_rissanen_out = min_rissanen;
    return GMM_OK;
}

}  // extern "C"
