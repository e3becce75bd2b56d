// host_math.cpp — GPU-free host numerics: M-step finalisation, constants
// (DxD inversion stays on the host: BASELINE.json north_star), seeding,
// Rissanen score, order reduction, and the worker team they run on.
// Semantics follow the reference (file:line cited per function); the code is
// written from scratch.
#include "host_math.h"

#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>

namespace gmm {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
int fail(int code, const std::string& msg) { g_err = msg; return code; }
const char* last_error_cstr() { return g_err.c_str(); }

// ---------------------------------------------------------------------------
// HostPool
// ---------------------------------------------------------------------------
static void cpu_relax() {
#if defined(__x86_64__) || defined(__i386__)
    __builtin_ia32_pause();
#endif
}

void HostPool::resize(int nthreads) {
    if (nthreads < 1) nthreads = 1;
    if (nthreads == size() && started_) return;
    stop();
    quit_.store(false);
    started_ = true;
    for (int i = 1; i < nthreads; i++) workers_.emplace_back([this] { worker(); });
}

void HostPool::run(int n, const std::function<void(int)>& fn) {
    if (n <= 0) return;
    if (workers_.empty() || n == 1) { for (int i = 0; i < n; i++) fn(i); return; }
    // Items are claimed by counting `remaining_` DOWN: a claim is valid iff the value it saw was positive, so a worker
    // still on its way out of the previous job's loop either sees <= 0 (before the store below) or a genuine item of
    // THIS job (after it) — there is no window in which a stale claim can be mistaken for a new one (an index
    // counted up against a separately published bound had one: found by gmm_host_pool_selftest).  Everything a
    // claimer reads is published before the store (release / acquire on `remaining_`).
    fn_ = &fn; n_ = n;
    done_.store(0, std::memory_order_relaxed);
    remaining_.store(n, std::memory_order_release);
    {
        std::lock_guard<std::mutex> lk(m_);
        gen_.fetch_add(1, std::memory_order_release);
    }
    cv_.notify_all();
    work();
    while (done_.load(std::memory_order_acquire) < n_) cpu_relax();
}

void HostPool::work() {
    for (;;) {
        const int r = remaining_.fetch_sub(1, std::memory_order_acq_rel);
        if (r <= 0) break;
        (*fn_)(r - 1);
        done_.fetch_add(1, std::memory_order_release);
    }
}

void HostPool::worker() {
    unsigned long long seen = gen_.load(std::memory_order_acquire);
    for (;;) {
        // spin for up to ~4 ms, then sleep
        const auto t0 = std::chrono::steady_clock::now();
        unsigned long long g;
        int spins = 0;
        while ((g = gen_.load(std::memory_order_acquire)) == seen && !quit_.load(std::memory_order_relaxed)) {
            cpu_relax();
            if ((++spins & 1023) == 0 && std::chrono::steady_clock::now() - t0 > std::chrono::milliseconds(4)) {
                std::unique_lock<std::mutex> lk(m_);
                cv_.wait(lk, [&] { return gen_.load(std::memory_order_acquire) != seen || quit_.load(); });
            }
        }
        if (quit_.load()) return;
        seen = g;
        work();
    }
}

void HostPool::stop() {
    if (!started_) return;
    {
        std::lock_guard<std::mutex> lk(m_);
        quit_.store(true);
    }
    cv_.notify_all();
    for (auto& t : workers_) t.join();
    workers_.clear();
    started_ = false;
}

// ---------------------------------------------------------------------------
// LU inverse without pivoting.  Same contract as invert_cpu
// (invert_matrix.cpp:25-101) / device invert (gaussian_kernel.cu:107-169):
// in place, no row exchanges, log|det| accumulated from the pivots.
// Doolittle factorisation A = L U (unit L), then A^-1 column by column.
// ---------------------------------------------------------------------------
template <class T>
void lu_inverse_nopivot(T* __restrict__ a, int n, T* logabsdet, T* __restrict__ w) {
    // Elimination applied to [A | I]: every inner loop is an axpy over a contiguous row (vectorises
    // without reassociation).  Forward pass leaves U in the upper triangle of `a` and L^-1 in `w`;
    // the backward pass turns `w` into U^-1 L^-1 = A^-1.
    for (int i = 0; i < n; i++)
        for (int j = 0; j < n; j++) w[i * n + j] = (i == j) ? T(1) : T(0);
    T ld = 0;
    for (int k = 0; k < n; k++) {
        const T piv = a[k * n + k];
        ld += std::log(std::fabs(piv));
        const T rp = T(1) / piv;
        const T* ak = a + k * n;
        const T* wk = w + k * n;
        for (int i = k + 1; i < n; i++) {
            const T l = a[i * n + k] * rp;
            T* ai = a + i * n;
            T* wi = w + i * n;
            for (int j = k + 1; j < n; j++) ai[j] -= l * ak[j];
            for (int j = 0; j <= k; j++) wi[j] -= l * wk[j];
        }
    }
    for (int k = n - 1; k >= 0; k--) {
        T* wk = w + k * n;
        for (int j = k + 1; j < n; j++) {
            const T u = a[k * n + j];
            const T* wj = w + j * n;
            for (int c = 0; c < n; c++) wk[c] -= u * wj[c];
        }
        const T rp = T(1) / a[k * n + k];
        for (int c = 0; c < n; c++) wk[c] *= rp;
    }
    for (int i = 0; i < n * n; i++) a[i] = w[i];
    *logabsdet = ld;
}
template void lu_inverse_nopivot<float>(float*, int, float*, float*);
template void lu_inverse_nopivot<double>(double*, int, double*, double*);

static const double kPi = 3.1415926535897931;   // gaussian.h:11

// constants_kernel (gaussian_kernel.cu:250-259): compute_constants (196-243)
// per cluster + compute_pi (172-193).  Inversion in double, results stored as
// float like the reference's clusters_t.
void constants_cluster(int k, int D, clusters_t* c) {
    double m[GMM_MAX_DIMENSIONS * GMM_MAX_DIMENSIONS], w[GMM_MAX_DIMENSIONS * GMM_MAX_DIMENSIONS];
    const float* R = c->R + (size_t)k * D * D;
    for (int i = 0; i < D * D; i++) m[i] = R[i];
    double ld;
    lu_inverse_nopivot<double>(m, D, &ld, w);
    float* Ri = c->Rinv + (size_t)k * D * D;
    for (int i = 0; i < D * D; i++) Ri[i] = (float)m[i];
    c->constant[k] = (float)(-D * 0.5 * std::log(2.0 * kPi) - 0.5 * ld);   // :241
}

// The same for a symmetric positive definite R through ONE factorisation: R = U U^T (U upper triangular, "reverse"
// Cholesky), W = U^-1 (upper triangular), Rinv = W^T W, ln det R = 2 sum ln U_ii — a third of the arithmetic of the
// LU inverse plus the separate factorisation of Rinv the tensor E-step's operand needs (W is handed to it directly).
// Returns false (nothing written) when R is not positive definite: the caller then takes the no-pivot LU path, whose
// semantics on such matrices are the reference's (invert_matrix.cpp:25-101).
bool constants_cluster_spd(int k, int D, clusters_t* c, double* W /* [D][D] out */) {
    double U[GMM_MAX_DIMENSIONS][GMM_MAX_DIMENSIONS];
    const float* R = c->R + (size_t)k * D * D;
    double ld = 0.0;
    for (int j = D - 1; j >= 0; j--) {
        double d = R[j * D + j];
        for (int m = j + 1; m < D; m++) d -= U[j][m] * U[j][m];
        if (!(d > 0.0) || !std::isfinite(d)) return false;
        const double piv = std::sqrt(d), rp = 1.0 / piv;
        U[j][j] = piv;
        ld += std::log(piv);
        for (int i = 0; i < j; i++) {
            double v = 0.5 * ((double)R[i * D + j] + (double)R[j * D + i]);
            for (int m = j + 1; m < D; m++) v -= U[i][m] * U[j][m];
            U[i][j] = v * rp;
        }
    }
    // W = U^-1 (upper triangular), column by column: W[i][j] = -(sum_{m=i+1..j} U[i][m] W[m][j]) / U[i][i]
    for (int j = 0; j < D; j++) {
        for (int i = D - 1; i > j; i--) W[i * D + j] = 0.0;
        W[j * D + j] = 1.0 / U[j][j];
        for (int i = j - 1; i >= 0; i--) {
            double v = 0.0;
            for (int m = i + 1; m <= j; m++) v -= U[i][m] * W[m * D + j];
            W[i * D + j] = v / U[i][i];
        }
    }
    float* Ri = c->Rinv + (size_t)k * D * D;
    for (int i = 0; i < D; i++)
        for (int j = i; j < D; j++) {                   // (W^T W)[i][j] = sum_{m <= i} W[m][i] W[m][j]
            double v = 0.0;
            for (int m = 0; m <= i; m++) v += W[m * D + i] * W[m * D + j];
            Ri[i * D + j] = (float)v;
            Ri[j * D + i] = (float)v;
        }
    c->constant[k] = (float)(-D * 0.5 * std::log(2.0 * kPi) - 0.5 * (2.0 * ld));   // gaussian_kernel.cu:241
    return true;
}

void mixing_weights(int K, clusters_t* c) {
    double sum = 0;                                                            // :176-181
    for (int k = 0; k < K; k++) sum += c->N[k];
    for (int k = 0; k < K; k++)                                                // :184-190
        c->pi[k] = (c->N[k] < 0.5f) ? 1e-10f : (float)(c->N[k] / sum);
}

void constants_from_R(int K, int D, clusters_t* c, HostPool& pool) {
    const std::function<void(int)> one = [&](int k) {
        double W[GMM_MAX_DIMENSIONS * GMM_MAX_DIMENSIONS];
        if (!constants_cluster_spd(k, D, c, W)) constants_cluster(k, D, c);     // not positive definite: the no-pivot LU semantics
    };
    if (K >= 8) pool.run(K, one);
    else for (int k = 0; k < K; k++) one(k);
    mixing_weights(K, c);
}

// Host side of the M-step (gaussian.cu:611-622 means, :663-679 covariance)
// together with the device-side rules of mstep_covariance1
// (gaussian_kernel.cu:658-675: zero if N < 1.0, += avgvar on the diagonal
// BEFORE the division).  Input statistics are taken about `shift`:
//   S0 = sum g, S1 = sum g (x - shift), S2 = sum g (x - shift)(x - shift)^T
// so that  sum g (x - mu)(x - mu)^T = S2 - S1 S1^T / S0  with mu = shift + S1/S0.
void finalize_cluster(const double* stats, const double* shift, int k, int D, clusters_t* c) {
    const int F = num_features(D);
    const double* s = stats + (size_t)k * F;
    const double S0 = s[0];
    const float Nf = (float)S0;
    c->N[k] = Nf;
    float* mu = c->means + (size_t)k * D;
    float* R = c->R + (size_t)k * D * D;
    double m[GMM_MAX_DIMENSIONS];
    for (int d = 0; d < D; d++) {
        m[d] = (S0 != 0.0) ? s[1 + d] / S0 : 0.0;
        mu[d] = (Nf > 0.5f) ? (float)(m[d] + shift[d]) : 0.0f;              // gaussian.cu:614-618
    }
    if (Nf > 0.5f) {
        const double inv = 1.0 / (double)Nf;
        for (int i = 0; i < D; i++)
            for (int j = 0; j <= i; j++) {
                double cov = (Nf >= 1.0f) ? s[feat2(D, i, j)] - m[i] * s[1 + j] : 0.0;   // kernel :658-668
                if (i == j) cov += c->avgvar[k];                                      // kernel :673-675
                const float v = (float)(cov * inv);                                   // gaussian.cu:664-667
                R[i * D + j] = v;
                R[j * D + i] = v;
            }
    } else {                                                                          // gaussian.cu:668-677
        for (int i = 0; i < D; i++)
            for (int j = 0; j < D; j++) R[i * D + j] = (i == j) ? 1.0f : 0.0f;
    }
}

void finalize_from_stats(const double* stats, const double* shift, int K, int D, clusters_t* c) {
    for (int k = 0; k < K; k++) finalize_cluster(stats, shift, k, D, c);
}

long long seed_event_index(int c, int K, long long N) {
    float seed = (K > 1) ? ((float)N - 1.0f) / ((float)K - 1.0f) : 0.0f;   // gaussian.cu:110-115
    return (long long)(int)((float)c * seed);                              // :120
}

void seed_from_moments(const double* sum_x, const double* sum_x2, long long N, int D, int K,
                       const float* seed_rows, clusters_t* c) {
    double total = 0;                                   // averageVariance, gaussian_kernel.cu:71-102
    for (int d = 0; d < D; d++) {
        const double mean = sum_x[d] / (double)N;
        total += sum_x2[d] / (double)N - mean * mean;
    }
    const float avgvar = (float)(total / D);
    for (int k = 0; k < K; k++) {                       // seed_clusters kernel :304-327
        for (int d = 0; d < D; d++) c->means[k * D + d] = seed_rows[k * D + d];
        float* R = c->R + (size_t)k * D * D;
        for (int i = 0; i < D; i++)
            for (int j = 0; j < D; j++) R[i * D + j] = (i == j) ? 1.0f : 0.0f;
        c->pi[k] = 1.0f / (float)K;
        c->N[k] = (float)N / (float)K;
        c->avgvar[k] = (float)(avgvar / 1e3);           // COVARIANCE_DYNAMIC_RANGE
    }
    HostPool serial(1);
    constants_from_R(K, D, c, serial);                  // gaussian.cu:404
    for (int k = 0; k < K; k++) c->N[k] = (float)(N / K);   // host seed_clusters: integer division, gaussian.cu:118
}

float rissanen(float loglik, int K, int D, long long N) {           // gaussian.cu:826
    return (float)(-loglik + 0.5 * (K * (1 + D + 0.5 * (D + 1) * D) - 1) * logf((float)N * D));
}
float em_epsilon(int D, long long N) {                              // gaussian.cu:458
    return (float)((1 + D + 0.5 * (D + 1) * D) * std::log((float)N * D) * 0.01);
}

// ---------------------------------------------------------------------------
// Order reduction (gaussian.cu:860-907).  Merge rule of add_clusters
// (gaussian.cu:1210-1252): weights N1/(N1+N2); merged mean; merged covariance
// = weighted (R_c + (mu - mu_c)(mu - mu_c)^T); pi and N add.  The merged
// constant uses log10(det) exactly as invert_cpu returns it
// (invert_matrix.cpp:61; quirk Q3) so that the merge SEQUENCE matches the
// reference.  Distance (cluster_distance :1203-1208):
//   N1*const1 + N2*const2 - N12*const12.
// ---------------------------------------------------------------------------
namespace {
struct Merged {
    float N, pi, constant;
    std::vector<float> means, R, Rinv;
};

void merge_pair(const clusters_t* c, int a, int b, int D, Merged& out) {
    out.means.resize(D); out.R.resize((size_t)D * D); out.Rinv.resize((size_t)D * D);
    const float wa = c->N[a] / (c->N[a] + c->N[b]);
    const float wb = 1.0f - wa;
    const float* ma = c->means + (size_t)a * D; const float* mb = c->means + (size_t)b * D;
    const float* Ra = c->R + (size_t)a * D * D; const float* Rb = c->R + (size_t)b * D * D;
    for (int i = 0; i < D; i++) out.means[i] = wa * ma[i] + wb * mb[i];
    for (int i = 0; i < D; i++)
        for (int j = i; j < D; j++) {
            float v = ((out.means[i] - ma[i]) * (out.means[j] - ma[j]) + Ra[i * D + j]) * wa;
            v += ((out.means[i] - mb[i]) * (out.means[j] - mb[j]) + Rb[i * D + j]) * wb;
            out.R[i * D + j] = v;
            out.R[j * D + i] = v;
        }
    out.pi = c->pi[a] + c->pi[b];
    out.N = c->N[a] + c->N[b];
    std::vector<float> work((size_t)D * D);
    out.Rinv = out.R;
    float lndet;
    lu_inverse_nopivot<float>(out.Rinv.data(), D, &lndet, work.data());
    const float log10det = (float)(lndet / std::log(10.0));
    out.constant = (float)((-D) * 0.5 * logf((float)(2 * kPi)) - 0.5 * log10det);
}

void move_cluster(clusters_t* c, int dst, int src, int D) {               // copy_cluster :1254-1264
    c->N[dst] = c->N[src]; c->pi[dst] = c->pi[src];
    c->constant[dst] = c->constant[src]; c->avgvar[dst] = c->avgvar[src];
    std::memmove(c->means + (size_t)dst * D, c->means + (size_t)src * D, sizeof(float) * D);
    std::memmove(c->R + (size_t)dst * D * D, c->R + (size_t)src * D * D, sizeof(float) * D * D);
    std::memmove(c->Rinv + (size_t)dst * D * D, c->Rinv + (size_t)src * D * D, sizeof(float) * D * D);
}
}  // namespace

int reduce_order(clusters_t* c, int K, int D, int* out_c1, int* out_c2, HostPool& pool) {
    for (int i = K - 1; i >= 0; i--)                                      // empties :866-874
        if (c->N[i] < 0.5f) {
            for (int j = i; j < K - 1; j++) move_cluster(c, j, j + 1, D);
            K--;
        }
    int best_a = 0, best_b = 1;
    if (K >= 2) {
        const int npairs = K * (K - 1) / 2;
        std::vector<float> dist(npairs);
        auto one_pair = [&](int p) {
            int a = 0, rem = p;                                           // p -> (a, b), a < b, row-major
            while (rem >= K - 1 - a) { rem -= K - 1 - a; a++; }
            const int b = a + 1 + rem;
            Merged m;
            merge_pair(c, a, b, D, m);
            dist[p] = c->N[a] * c->constant[a] + c->N[b] * c->constant[b] - m.N * m.constant;
        };
        if (npairs >= 64) pool.run((npairs + 15) / 16, [&](int t) { for (int p = t * 16; p < npairs && p < t * 16 + 16; p++) one_pair(p); });
        else for (int p = 0; p < npairs; p++) one_pair(p);
        float best = 0.0f;
        int p = 0;
        for (int a = 0; a < K; a++)                                       // first strict minimum :882-894
            for (int b = a + 1; b < K; b++, p++)
                if ((a == 0 && b == 1) || dist[p] < best) { best = dist[p]; best_a = a; best_b = b; }
        Merged m;
        merge_pair(c, best_a, best_b, D, m);                              // :899-907
        c->N[best_a] = m.N; c->pi[best_a] = m.pi; c->constant[best_a] = m.constant;
        c->avgvar[best_a] = c->avgvar[0];
        std::memcpy(c->means + (size_t)best_a * D, m.means.data(), sizeof(float) * D);
        std::memcpy(c->R + (size_t)best_a * D * D, m.R.data(), sizeof(float) * D * D);
        std::memcpy(c->Rinv + (size_t)best_a * D * D, m.Rinv.data(), sizeof(float) * D * D);
        for (int i = best_b; i < K - 1; i++) move_cluster(c, i, i + 1, D);
    }
    if (out_c1) *out_c1 = best_a;
    if (out_c2) *out_c2 = best_b;
    return K - 1;                                                         // loop decrement, gaussian.cu:479
}

int epack_stride(int D) {
    const int coef_off = (D + 3) & ~3;
    return (coef_off + D * (D + 1) / 2 + 1 + 3) & ~3;
}

// E-step parameters of estep1 (gaussian_kernel.cu:412-423) pre-combined:
// the full D x D loop of :435-439 equals sum_i dx_i (Rinv_ii dx_i + sum_{j>i}
// (Rinv_ij + Rinv_ji) dx_j); constant + logf(pi) is the additive term of :442.
void build_epack(int K, int D, const clusters_t* c, float* out) {
    const int stride = epack_stride(D), coef_off = (D + 3) & ~3;
    std::memset(out, 0, sizeof(float) * (size_t)K * stride);
    for (int k = 0; k < K; k++) {
        float* p = out + (size_t)k * stride;
        const float* Ri = c->Rinv + (size_t)k * D * D;
        for (int d = 0; d < D; d++) p[d] = c->means[(size_t)k * D + d];
        int idx = coef_off;
        for (int i = 0; i < D; i++)
            for (int j = i; j < D; j++)
                p[idx++] = (i == j) ? Ri[i * D + i] : Ri[i * D + j] + Ri[j * D + i];
        p[idx] = c->constant[k] + logf(c->pi[k]);
    }
}

}  // namespace gmm

// ---------------------------------------------------------------------------
// extern "C" wrappers (include/gmm.h, "host-only numerics")
// ---------------------------------------------------------------------------
namespace gmm { const char* last_error_cstr(); }

extern "C" {

const char* gmm_last_error(void) { return gmm::last_error_cstr(); }

int gmm_host_invert(float* data, int n, float* log_det, int use_log10) {
    if (!data || !log_det || n < 1 || n > GMM_MAX_DIMENSIONS) return gmm::fail(GMM_ERR_ARG, "gmm_host_invert: bad argument");
    std::vector<float> work((size_t)n * n);
    float ln;
    gmm::lu_inverse_nopivot<float>(data, n, &ln, work.data());
    *log_det = use_log10 ? (float)(ln / std::log(10.0)) : ln;
    return GMM_OK;
}

long long gmm_stats_len(int K, int D) { return (long long)K * gmm::num_features(D) + 1; }

int gmm_host_finalize(const double* stats, const double* shift, int K, int D, clusters_t* inout) {
    if (!stats || !shift || !inout || K < 1 || K > GMM_MAX_CLUSTERS || D < 1 || D > GMM_MAX_DIMENSIONS)
        return gmm::fail(GMM_ERR_ARG, "gmm_host_finalize: bad argument");
    gmm::HostPool serial(1);
    gmm::finalize_from_stats(stats, shift, K, D, inout);
    gmm::constants_from_R(K, D, inout, serial);
    return GMM_OK;
}

float gmm_host_rissanen(float loglik, int K, int D, long long N) { return gmm::rissanen(loglik, K, D, N); }
float gmm_host_epsilon(int D, long long N) { return gmm::em_epsilon(D, N); }

int gmm_host_reduce_order(clusters_t* clusters, int* K, int D, int* c1, int* c2) {
    if (!clusters || !K || *K < 1 || D < 1 || D > GMM_MAX_DIMENSIONS) return gmm::fail(GMM_ERR_ARG, "gmm_host_reduce_order: bad argument");
    gmm::HostPool serial(1);
    *K = gmm::reduce_order(clusters, *K, D, c1, c2, serial);
    return GMM_OK;
}

// Self-test of HostPool (tests/test_host.py): `jobs` back-to-back parallel loops of n items on `threads` threads, every
// item must run exactly once per job.  Returns 0 when it did.
int gmm_host_pool_selftest(int threads, int jobs, int n) {
    if (threads < 1 || jobs < 1 || n < 0) return gmm::fail(GMM_ERR_ARG, "gmm_host_pool_selftest: bad argument");
    gmm::HostPool pool(threads);
    std::vector<std::atomic<int>> hits((size_t)(n > 0 ? n : 1));
    for (auto& h : hits) h.store(0);
    for (int j = 0; j < jobs; j++) {
        const int m = (j % 3 == 0) ? n : (j % 3 == 1 ? (n + 1) / 2 : 1);
        const std::function<void(int)> fn = [&](int i) { hits[(size_t)i].fetch_add(1, std::memory_order_relaxed); };
        pool.run(m, fn);
        for (int i = 0; i < n; i++) {
            const int want = i < m ? 1 : 0;
            if (hits[(size_t)i].exchange(0) != want) return gmm::fail(GMM_ERR_STATE, "gmm_host_pool_selftest: an item ran the wrong number of times");
        }
        if (j % 64 == 63) pool.resize(1 + (j / 64) % threads);          // exercise team re-creation as well
        if (j % 200 == 199) std::this_thread::sleep_for(std::chrono::milliseconds(6));   // let the workers fall asleep once in a while
    }
    return GMM_OK;
}

void gmm_shard_range(long long n_global, int nranks, int rank, long long* begin, long long* count) {
    const long long per = n_global / nranks;                  // gaussian.cu:348-352 (Q6 fixed)
    if (begin) *begin = per * rank;
    if (count) *count = (rank == nranks - 1) ? per + n_global % nranks : per;
}

}  // extern "C"
