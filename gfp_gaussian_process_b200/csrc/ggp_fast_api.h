// ggp_fast_api.h — what ggp_b200.cu (strict translation unit, -fmad=false) calls in ggp_fast.cu (fast likelihood kernels,
// -fmad=true).  Internal to the library.
#pragma once
#include <cuda_runtime.h>

#include "ggp_types.cuh"

#define GGP_FAST_DEFAULT_NODES 6   // exact to rounding while the exponent varies by <= 0.5 over a time step (GgpFastLmax)

// quadrature orders the fast kernels are instantiated for
bool ggp_fast_supported_nodes(int n_nodes);
// bytes of one entry of the constants table (GgpFastConsts<double, N>)
size_t ggp_fast_consts_bytes(int n_nodes);
// the (parameters, dt)-only constants of every (vector of the chunk, distinct time step) pair into
// ktab[(v - A.v0) * n_dt + d]: one tiny launch per vector chunk
cudaError_t ggp_fast_consts_launch(const GgpFwdArgs& A, const double* dt_values, int n_dt, void* ktab, int n_nodes, cudaStream_t stream);
// one generation (or one upload chunk of it) of the likelihood for the vectors of A; grid.y = A.v_count.
// invalid [n_vec]: set to 1 for a vector whose evaluation left the quadrature's validity range or met a NaN term
// (the caller re-runs it on the strict path).  Same partial / state / cell_ll conventions as the strict kernels.
cudaError_t ggp_fast_loglik_launch(const GgpDevForest& F, const GgpFwdArgs& A, const void* ktab, int* invalid, int n_nodes,
                                   cudaStream_t stream);
