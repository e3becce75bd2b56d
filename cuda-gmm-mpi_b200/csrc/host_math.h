// host_math.h — GPU-free host numerics of the engine (internal C++ API).
// The extern "C" wrappers of include/gmm.h live in host_math.cpp.
#pragma once
#include <atomic>
#include <condition_variable>
#include <cstddef>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>
#include "../../include/gmm.h"

namespace gmm {

void set_error(const std::string& msg);          // thread-local, read by gmm_last_error()
int  fail(int code, const std::string& msg);     // set_error + return code

// Number of per-cluster sufficient statistics: 1 + D + D(D+1)/2.
inline int num_features(int D) { return 1 + D + D * (D + 1) / 2; }
// Index of the second-moment feature (i >= j) inside a cluster's feature row.
inline int feat2(int D, int i, int j) { return 1 + D + i * (i + 1) / 2 + j; }

// In-place inverse by LU factorisation WITHOUT pivoting (the semantics of
// invert_cpu, invert_matrix.cpp:25-101, and of the device `invert`,
// gaussian_kernel.cu:107-169).  Returns sum log|u_ii| in *logabsdet (natural
// log).  T = float or double.
template <class T> void lu_inverse_nopivot(T* a, int n, T* logabsdet, T* work /* n*n */);

// Persistent worker team for the host's loops over clusters (K independent clusters, a few microseconds each).
// The workers SPIN on a generation counter for a few milliseconds after each job — an EM iteration hands them the
// next one within that window — and only then block on a condition variable.  An OpenMP parallel region costs a
// futex wake-up per thread and iteration when the runtime's wait policy is passive (torchrun exports OMP_NUM_THREADS=1
// and the measured finalisation went from 0.05 ms to 0.33 ms per iteration at 2 ranks).  HostPool(1) starts no thread:
// run() is then a plain serial loop.
class HostPool {
public:
    explicit HostPool(int nthreads) { resize(nthreads); }
    ~HostPool() { stop(); }
    int size() const { return (int)workers_.size() + 1; }
    void resize(int nthreads);
    // fn(i) for i in [0, n), spread dynamically over the team (the caller takes part); returns when all are done
    void run(int n, const std::function<void(int)>& fn);
private:
    void work();
    void worker();
    void stop();
    std::vector<std::thread> workers_;
    std::mutex m_;
    std::condition_variable cv_;
    std::atomic<unsigned long long> gen_{0};
    std::atomic<int> remaining_{0}, done_{0};
    std::atomic<bool> quit_{false};
    const std::function<void(int)>* fn_ = nullptr;
    int n_ = 0;
    bool started_ = false;
};

// N, means, R of every cluster from reduced statistics (finalize_cluster in a loop).
void finalize_from_stats(const double* stats, const double* shift, int K, int D, clusters_t* c);

// constants_kernel semantics on host arrays: Rinv, constant (ln det), pi.  The clusters run on `pool` when K >= 8.
void constants_from_R(int K, int D, clusters_t* c, HostPool& pool);
// The two parts of constants_from_R, for callers that run their own loop over the clusters:
// inverse + constant of one cluster, and the mixing weights pi (needs every N[k]).
void constants_cluster(int k, int D, clusters_t* c);
// Same results for a symmetric positive definite R from one (reverse) Cholesky factorisation; also returns the
// upper-triangular W with Rinv = W^T W.  false = not positive definite, nothing written (use constants_cluster).
bool constants_cluster_spd(int k, int D, clusters_t* c, double* W);
// N, mean and covariance of ONE cluster from the packed statistics (the loop body of finalize_from_stats).
void finalize_cluster(const double* stats, const double* shift, int k, int D, clusters_t* c);
void mixing_weights(int K, clusters_t* c);

// Seeding from global column sums (double): sum x, sum x^2 over all N events,
// and the K seed rows (already gathered).  gaussian_kernel.cu:269-328,
// gaussian.cu:108-123.
void seed_from_moments(const double* sum_x, const double* sum_x2, long long N, int D, int K,
                       const float* seed_rows /* [K][D] */, clusters_t* c);
// Row index of seed event c (gaussian.cu:110-120: (int)(c*seed), seed in float).
long long seed_event_index(int c, int K, long long N);

float rissanen(float loglik, int K, int D, long long N);
float em_epsilon(int D, long long N);

// One order-reduction step (gaussian.cu:860-907).  Returns new K.  The K(K-1)/2 trial merges run on `pool`
// (16 pairs per item) when there are at least 64 of them.
int reduce_order(clusters_t* c, int K, int D, int* c1, int* c2, HostPool& pool);

// Packed E-step parameters for the SIMT kernel: per cluster
//   [ mean(D) | c_ii, 2c_ij (j>i) row by row (D(D+1)/2) | constant + ln(pi) ] padded to stride.
int  epack_stride(int D);
void build_epack(int K, int D, const clusters_t* c, float* out);

}  // namespace gmm
