// kernels_tc.cuh — tcgen05 (5th-generation tensor core) path of the EM hot
// path.  Interface used by gmm_api.cu; implementation in kernels_tc.cu.
#pragma once
#include <cuda_runtime.h>
#include "../../include/gmm.h"

namespace gmm {

struct TcState;

// Shapes the tensor-core kernels cover (independently for the two steps).
bool tc_mstep_supported(int D, int K);
bool tc_estep_supported(int D, int K);

// memb_pitch: row pitch (in floats) of the cluster-major responsibilities buffer AND of the SoA event copy.
int  tc_create(TcState** out, const float* d_x_aos, const float* d_x_soa, int n, int D, int Kmax, float* d_memb, size_t memb_pitch,
               int num_sms, cudaStream_t stream);
void tc_destroy(TcState*);
// Centre/scale used inside the tensor kernels: z = (x - shift) * inv_scale, both rounded to
// float; `shift` is updated in place to the float-rounded values actually used.  xmin / xmax: per-dimension extremes
// of the WHOLE data set (all ranks): they fix the power-of-two quanta of the M-step's fixed-point operand parts.
int  tc_set_shift_scale(TcState*, double* shift, const double* scale, const double* xmin, const double* xmax, cudaStream_t stream);
// True once the quanta are set and the data range fits the fixed-point budget (|z| <= 64 global standard deviations);
// otherwise the caller uses the FP64 SIMT M-step.
bool tc_mstep_ready(const TcState*);
// False when an event lies beyond 2^14 global standard deviations (its standardised coordinates would overflow FP16).
bool tc_estep_range_ok(const TcState*);
// The tensor E-step operand of the host parameters in three steps, so that the caller can fuse the per-cluster work
// with its own per-cluster finalisation in ONE parallel loop: begin (serial), cluster k in [0, tc_params_padded)
// (independent, thread safe; returns 0 or a defect code to be max-reduced), commit (serial: error report or H2D of
// the operand).
int  tc_params_begin(TcState*, int K, cudaStream_t stream);
int  tc_params_padded(const TcState*, int K);
int  tc_params_cluster(TcState*, const clusters_t* host, int k, int K);
// The same with the upper-triangular factor W (Rinv = W^T W, double, row-major [D][D]) supplied by the caller
// (constants_cluster_spd): no second factorisation of the inverse.
int  tc_params_cluster_w(TcState*, const clusters_t* host, int k, int K, const double* W);
int  tc_params_commit(TcState*, int K, int bad, cudaStream_t stream);
int  tc_launch_estep(TcState*, int K, double* d_ll, cudaStream_t stream);
// Device-side M-step finalisation: reduced statistics -> parameter set `d_set` (floats, tc_param_set_floats(); arrays at
// tc_param_set_off(which = 0 N, 1 pi, 2 constant, 3 means, 4 R, 5 Rinv), stride Kmax) + the E-step operand, no host round
// trip.  d_ll[0] receives the log-likelihood slot of the statistics.  d_bad[0] = first iteration (`iter`) that met a cluster
// the host path must handle (-1: none; later launches then return immediately), d_bad[1] = its code (1 not positive
// definite, 2 outside FP16, 4 statistics not finite).
bool tc_finalize_supported(const TcState*, int K);
size_t tc_param_set_floats(int Kmax, int D);
size_t tc_param_set_off(int Kmax, int D, int which);
// fault_iter: the launch with iter == fault_iter reports code 1 although nothing is wrong (-1: never; test hook).
int  tc_launch_finalize(TcState*, int K, const double* d_stats, const float* d_avgvar, float* d_set, double* d_ll, int* d_bad, int iter,
                        int fault_iter, cudaStream_t stream);
// Accumulates sum_n g[k][n] * phi_f(x_n - shift) into d_stats[k*F + f] (double, original units).
int  tc_launch_mstep(TcState*, int K, double* d_stats, cudaStream_t stream);

}  // namespace gmm
