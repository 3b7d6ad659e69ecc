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

// ---- gradient (forward mode over the fast step, ggp_dual.cuh) ----
#define GGP_GRAD_D 1   // parameter directions carried by one thread
// the parameter indices to differentiate along; block b of a vector carries directions idx[b * GGP_GRAD_D ..]
struct GgpGradDirs {
    int32_t n;
    int32_t idx[GGP_NP];
};
// bytes of one entry of the gradient's constants table (GgpFastConsts<GgpDual<GGP_GRAD_D>, N>)
size_t ggp_fast_grad_consts_bytes(int n_nodes);
// the dual constants of every (vector of the chunk, direction block, distinct time step) into
// ktab[((v - A.v0) * n_blocks + b) * n_dt + d], n_blocks = ceil(G.n / GGP_GRAD_D); A.params must be a device array
cudaError_t ggp_fast_grad_consts_launch(const GgpFwdArgs& A, const GgpGradDirs& G, const double* dt_values, int n_dt, void* ktab,
                                        int n_nodes, cudaStream_t stream);
// one generation (or one upload chunk of it) of the value and the directional derivatives; grid.y = A.v_count * n_blocks.
// A.state holds 14 (1 + GGP_GRAD_D) rows of A.v_count * n_blocks * n_cells; A.partial [A.v_count * n_blocks * (1 + GGP_GRAD_D)]
// [n_partial]: row (v * n_blocks + b) * (1 + GGP_GRAD_D) + j is the value (j = 0) or tangent j - 1.  invalid as for the likelihood.
cudaError_t ggp_fast_grad_launch(const GgpDevForest& F, const GgpFwdArgs& A, const GgpGradDirs& G, const void* ktab, int* invalid,
                                 int n_nodes, cudaStream_t stream);

// ---- Hessian (forward mode over the fast step with GgpTaylor2, second-order Taylor numbers along one direction) ----
// the evaluations of one vector a launch runs: evaluation e steps along s_a e_a + s_b e_b with a = a[e], b = b[e] parameter
// indices (a == b: s_a e_a) and s = ggp_hess_scale(p) of the vector's parameters; the host enumerates the n (n + 1) / 2 pairs of
// a direction set and hands them over in ranges
#define GGP_HESS_MAX_EVALS (GGP_NP * (GGP_NP + 1) / 2)
struct GgpHessDirs {
    int32_t n;
    int8_t a[GGP_HESS_MAX_EVALS], b[GGP_HESS_MAX_EVALS];
};
// bytes of one entry of the Hessian's constants table (GgpFastConsts<GgpTaylor2, N>)
size_t ggp_fast_hess_consts_bytes(int n_nodes);
// as ggp_fast_grad_consts_launch with evaluation e in place of direction block b: ktab[((v - A.v0) * H.n + e) * n_dt + d]
cudaError_t ggp_fast_hess_consts_launch(const GgpFwdArgs& A, const GgpHessDirs& H, const double* dt_values, int n_dt, void* ktab,
                                        int n_nodes, cudaStream_t stream);
// as ggp_fast_grad_launch with H.n evaluations per vector and 3 results each: A.state holds 14 x 3 rows of
// A.v_count * H.n * n_cells; partial row (v * H.n + e) * 3 + j is the value (j = 0), g.u (1) and u^T H u (2)
cudaError_t ggp_fast_hess_launch(const GgpDevForest& F, const GgpFwdArgs& A, const GgpHessDirs& H, const void* ktab, int* invalid,
                                 int n_nodes, cudaStream_t stream);
