// ggp_kernels.cuh — what the sm_100a kernels of the strict unit share (FP64, strict rounding): the math tables
// (exp/log/pow/Dawson, 14 kB) staged in shared memory, the one-thread-per-element scratch layout, the fill and fixed-order
// reduction kernels, combine_predictions (predictions.h:466) and the self-test kernels.
//
// The reference walks each tree depth first on one core.  Here the forest is stored in generation order
// ("slots": all roots, then all their daughters, ...; inside a generation cells are sorted by length so
// the lanes of a warp run the same number of time points) and one launch handles one generation; the
// likelihood and prediction passes are in ggp_coop_kernels.cuh (four warps per 32 cells).  The per-cell
// log-evidence is reduced in a fixed order (warp shuffle -> one partial per 32 cells -> one value per vector),
// so results are reproducible run to run.
#pragma once
#include "ggp_tables_data.h"
#include "ggp_cell.cuh"

#define GGP_BLOCK 128

__device__ const GgpMathTables g_ggp_tables = GGP_MATH_TABLES_INIT;

// dynamic shared memory of the one-thread-per-element kernels (joint prep, propagate self-test): [math tables][per-thread scratch, GGP_SCRATCH x GGP_BLOCK doubles]
#define GGP_SMEM_BYTES (sizeof(GgpMathTables) + (size_t)GGP_SCRATCH * GGP_BLOCK * sizeof(double))

__device__ __forceinline__ GgpScratch ggp_thread_scratch() {
    GgpScratch S;
    S.base = reinterpret_cast<double*>(ggp_smem + sizeof(GgpMathTables)) + threadIdx.x;
    S.stride = GGP_BLOCK;
    return S;
}

__device__ __forceinline__ void ggp_stage_tables(GgpMathTables* sm) {
    const uint64_t* src = reinterpret_cast<const uint64_t*>(&g_ggp_tables);
    uint64_t* dst = reinterpret_cast<uint64_t*>(sm);
    for (int i = threadIdx.x; i < (int)(sizeof(GgpMathTables) / 8); i += blockDim.x) dst[i] = src[i];
    __syncthreads();
}

// 64-bit fill (cudaMemsetAsync may be routed through a copy engine and queue behind a streamed upload)
__global__ void __launch_bounds__(256) ggp_fill64_kernel(unsigned long long* __restrict__ p, unsigned long long v, size_t n) {
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) p[i] = v;
}

// one value per vector from the per-block partials, fixed order.  A thread's loads are issued 8 at a time ahead of its adds
// (the adds keep their order): one add per dependent load left the kernel waiting on memory latency ~20 times in a row
__global__ void __launch_bounds__(256) ggp_reduce_kernel(const double* __restrict__ partial, int n_partial,
                                                         double* __restrict__ out) {
    __shared__ double sm[256];
    const double* p = partial + (int64_t)blockIdx.x * n_partial;
    double s = 0.0;
    int i = threadIdx.x;
    for (; i + 7 * 256 < n_partial; i += 8 * 256) {
        double v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = p[i + k * 256];
#pragma unroll
        for (int k = 0; k < 8; ++k) s = s + v[k];
    }
    for (; i < n_partial; i += 256) s = s + p[i];
    sm[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sm[threadIdx.x] = sm[threadIdx.x] + sm[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[blockIdx.x] = sm[0];
}

__global__ void __launch_bounds__(GGP_BLOCK) ggp_combine_kernel(int64_t n_ctp, const double* __restrict__ fwd,
                                                                const double* __restrict__ bwd,
                                                                const int32_t* __restrict__ comb_seg,
                                                                const double* __restrict__ params,
                                                                double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * GGP_BLOCK + threadIdx.x;
    if (i >= n_ctp) return;
    ggp_ctp_combine(fwd + 20 * i, bwd + 20 * i, params + GGP_NP * comb_seg[i], out + 20 * i);
}

// ---- self-test kernels (ggp_math_eval / ggp_propagate_eval) -------------------------------------
__global__ void __launch_bounds__(GGP_BLOCK) ggp_math_kernel(int fn, int64_t n, const double* __restrict__ x,
                                                             const double* __restrict__ y, double* __restrict__ out) {
    GgpMathTables& T = *reinterpret_cast<GgpMathTables*>(ggp_smem);
    ggp_stage_tables(&T);
    const int64_t i = (int64_t)blockIdx.x * GGP_BLOCK + threadIdx.x;
    if (i >= n) return;
    double r;
    switch (fn) {
        case 0: r = ggp_exp(x[i], &T); break;
        case 1: r = ggp_log(x[i], &T); break;
        case 2: r = ggp_pow(x[i], y[i], &T); break;
        case 3: r = ggp_dawson(x[i], &T); break;
        default: r = x[i] / ggp_divisor(y[i]); break;
    }
    out[i] = r;
}

__global__ void __launch_bounds__(GGP_BLOCK) ggp_propagate_kernel(int64_t n, const double* __restrict__ state14,
                                                                  const double* __restrict__ dt,
                                                                  const double* __restrict__ p7, double* __restrict__ out14,
                                                                  double* __restrict__ cross16) {
    GgpMathTables& T = *reinterpret_cast<GgpMathTables*>(ggp_smem);
    ggp_stage_tables(&T);
    const int64_t i = (int64_t)blockIdx.x * GGP_BLOCK + threadIdx.x;
    if (i >= n) return;
    GgpState s;
#pragma unroll
    for (int k = 0; k < 4; ++k) s.m[k] = state14[14 * i + k];
#pragma unroll
    for (int k = 0; k < 10; ++k) s.c[k] = state14[14 * i + 4 + k];
    GgpOuParams p = {p7[7 * i], p7[7 * i + 1], p7[7 * i + 2], p7[7 * i + 3], p7[7 * i + 4], p7[7 * i + 5], p7[7 * i + 6]};
    double cr[16];
    ggp_propagate_impl(s, dt[i], p, &T, ggp_thread_scratch(), cross16 ? cr : nullptr);
#pragma unroll
    for (int k = 0; k < 4; ++k) out14[14 * i + k] = s.m[k];
#pragma unroll
    for (int k = 0; k < 10; ++k) out14[14 * i + 4 + k] = s.c[k];
    if (cross16) {
#pragma unroll
        for (int k = 0; k < 16; ++k) cross16[16 * i + k] = cr[k];
    }
}

// ---- FP64 pipe peak (roofline denominator; MEASURED_PEAKS.json has no FP64 figure) ----------------
// register-resident DFMA chains: 8 independent accumulators per thread, 2 flop per DFMA
__global__ void __launch_bounds__(256) ggp_fp64_peak_kernel(int iters, double a, double b, double* __restrict__ out) {
    double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; ++i) {
        x0 = __fma_rn(x0, a, b); x1 = __fma_rn(x1, a, b); x2 = __fma_rn(x2, a, b); x3 = __fma_rn(x3, a, b);
        x4 = __fma_rn(x4, a, b); x5 = __fma_rn(x5, a, b); x6 = __fma_rn(x6, a, b); x7 = __fma_rn(x7, a, b);
    }
    const double r = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    if (r == 12345.678) out[0] = r;   // never true; keeps the chains alive
}
