// ggp_fast_api.h — what ggp_b200.cu (strict translation unit, -fmad=false) calls in ggp_fast.cu (fast likelihood kernels,
// -fmad=true).  Internal to the library.  One kernel family serves the log-likelihood (plan order 0), its gradient (1) and its
// Hessian (2); the plan (GgpEvalPlan, ggp_types.cuh) says which, and which evaluations of every vector a launch runs
// (plan.n_run of them, picked by plan.select).
#pragma once
#include <cuda_runtime.h>

#include "ggp_types.cuh"

#define GGP_FAST_DEFAULT_NODES 6   // exact to rounding while the exponent varies by <= 0.5 over a time step (GgpFastLmax)

// quadrature orders the fast kernels are instantiated for
bool ggp_fast_supported_nodes(int n_nodes);
// bytes of one entry of the plan's constants table (GgpFastConsts<scalar, N>)
size_t ggp_fast_consts_bytes(const GgpEvalPlan& plan, int n_nodes);
// the (parameters, dt)-only constants of every (vector of the chunk, evaluation, distinct time step) into
// ktab[((v - A.v0) * plan.n_run + e) * n_dt + d]: one tiny launch per vector chunk.  Derivatives read device parameters
cudaError_t ggp_fast_consts_launch(const GgpFwdArgs& A, const GgpEvalPlan& plan, const double* dt_values, int n_dt, void* ktab,
                                   int n_nodes, cudaStream_t stream);
// one generation (or one upload chunk of it) of the plan's evaluations for the vectors of A; grid.y = A.v_count * plan.n_run.
// A.state holds 14 x C rows of A.v_count * plan.n_run * n_cells, C = plan.comps(); partial row (v * plan.n_run + e) * C + j is
// the value (j = 0), g.u (1) or u^T H u (2) of the evaluation's direction u.  Order 0 writes A.cell_ll, the same partial / state
// / cell_ll conventions as the strict kernels; order 1 writes, when A.cell_ll is not null, every cell's value and g.u into
// A.cell_ll[((v - A.v0) * plan.n_run + e) * 2 + j][n_cells] (caller's cell order).  invalid [n_vec]: set to 1 for a vector whose evaluation left the quadrature's
// validity range or met a NaN term (the caller re-runs it).
cudaError_t ggp_fast_loglik_launch(const GgpDevForest& F, const GgpFwdArgs& A, const GgpEvalPlan& plan, const void* ktab, int* invalid,
                                   int n_nodes, cudaStream_t stream);
// out[r][n_trees] = sum of rows[r][c] over the cells c = tree_cells[tree_off[t] .. tree_off[t + 1]) of tree t, in that order, for
// r < n_rows; the bits depend on the tree's cell list only
cudaError_t ggp_tree_sum_launch(const double* rows, int64_t n_cells, int64_t n_rows, const int64_t* tree_off, const int32_t* tree_cells,
                                int32_t n_trees, double* out, cudaStream_t stream);
