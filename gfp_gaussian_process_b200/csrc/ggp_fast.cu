// ggp_fast.cu — the FAST likelihood kernels (ggp_fast.cuh): one thread per (cell, parameter vector), one launch per
// generation, mother -> daughter hand-over through the same SoA state buffer and the same fixed-order reduction as the strict
// path.  Compiled with FMA contraction ON (-fmad=true); nothing of the strict math is included here.
//
// What depends on (parameters, dt) only - exp(-b t), the OU noise terms, the quadrature nodes t xi_j and exp(-+gq t xi_j):
// 16 + 16 N doubles, pre-multiplied for the quadrature sums - is tabulated once per (vector, distinct dt of the forest) by ggp_fast_consts_kernel; the forest stores
// the table index of every time point (2 bytes per point instead of the 8-byte time stamp).  Tables of up to
// GGP_FAST_SMEM_DT entries are staged in shared memory, larger ones are read through L1.
//
// Build: nvcc -std=c++17 -O3 -fmad=true -gencode arch=compute_100a,code=sm_100a -lineinfo -c
#include "ggp_fast_api.h"
#include "ggp_fast.cuh"

#define GGP_FAST_BLOCK 128
#define GGP_FAST_SMEM_DT 16

template <int N>
__global__ void __launch_bounds__(128) ggp_fast_consts_kernel(const GgpFwdArgs A, const double* __restrict__ dt_values, int n_dt,
                                                              GgpFastConsts<double, N>* __restrict__ ktab) {
    const int i = blockIdx.x * 128 + threadIdx.x;
    if (i >= n_dt * A.v_count) return;
    const int v = i / n_dt, d = i - v * n_dt;
    const double* p = A.params ? A.params + (int64_t)(A.v0 + v) * GGP_NP : A.inline_params + (A.v0 + v) * GGP_NP;
    GgpFastConsts<double, N> K;
    ggp_fast_consts(K, dt_values[d], p[0], p[1], p[2], p[3], p[4], p[5], p[6], GgpGLRule<N>());
    ktab[i] = K;
}

template <int N, bool ONE>
struct GgpFastConstsTable {
    const GgpFastConsts<double, N>* tab;   // this vector's entries
    const uint16_t* __restrict__ idx;
    // ONE: the forest has a single distinct time step (a fixed acquisition interval): no index to read.  The zero comes out of
    // an opaque instruction: with a literal the compiler hoists the entry's 16 + 16 N loads out of the step loop (1.5 kB of spills)
    __device__ __forceinline__ const GgpFastConsts<double, N>& at(int64_t k, int64_t) const {
        if (ONE) {
            int z;
            asm volatile("mov.s32 %0, 0;" : "=r"(z));
            return tab[z];
        }
        // (reading the index one step ahead - a register across the step, or across the measurement update only - was measured
        // slower: 0.67 / 0.63 vs 0.61 ms; at 168 registers the extra live value is spilled right behind its load)
        return tab[idx[k]];
    }
};

// The register allocation is made for 3 resident blocks per SM: 2 / 3 / 4 blocks (242 / 168 / 128 registers) measured
// 0.777 / 0.752 / 0.864 ms on configs[1] with 6 nodes.
// TAB 0: the constants table is read through L1; 1: it fits the block's shared copy (n_dt <= GGP_FAST_SMEM_DT): shared-memory loads
// with known address space; 2: one entry (n_dt == 1), shared, and the per-point index is not read at all (its load was the
// kernel's one exposed memory latency: the table address of a step depends on it)
template <int N, int TAB>
__global__ void __launch_bounds__(GGP_FAST_BLOCK, 3) ggp_fast_loglik_kernel(const GgpDevForest F, const GgpFwdArgs A,
                                                                        const GgpFastConsts<double, N>* __restrict__ ktab,
                                                                        int* __restrict__ invalid) {
    __shared__ double sp[GGP_NP];
    __shared__ double red[GGP_FAST_BLOCK / 32];
    constexpr bool SMEM = TAB != 0;
    __shared__ GgpFastConsts<double, N> ks[TAB == 1 ? GGP_FAST_SMEM_DT : 1];
    const int lane_slot = blockIdx.x * GGP_FAST_BLOCK + threadIdx.x;
    const bool active = lane_slot < A.n_slots;
    const int slot = A.slot0 + (active ? lane_slot : 0);
    const int v = blockIdx.y;
    if (threadIdx.x < GGP_NP)
        sp[threadIdx.x] = A.params ? A.params[(int64_t)(A.v0 + v) * GGP_NP + threadIdx.x] : A.inline_params[(A.v0 + v) * GGP_NP + threadIdx.x];
    const GgpFastConsts<double, N>* kv = ktab + (int64_t)v * F.n_dt;
    if (SMEM) {
        const double* src = reinterpret_cast<const double*>(kv);
        double* dst = reinterpret_cast<double*>(ks);
        for (int i = threadIdx.x; i < F.n_dt * (int)(sizeof(GgpFastConsts<double, N>) / sizeof(double)); i += GGP_FAST_BLOCK) dst[i] = src[i];
    }
    __syncthreads();
    double own = 0.0;
    if (active) {
        const int64_t vstride = (int64_t)A.v_count * F.n_cells;
        const int64_t vbase = (int64_t)v * F.n_cells;
        const int parent = F.s_parent[slot];
        GgpFastState<double> s;
        if (parent >= 0) {
#pragma unroll
            for (int k = 0; k < 4; ++k) s.m[k] = A.state[k * vstride + vbase + parent];
#pragma unroll
            for (int k = 0; k < 10; ++k) s.c[k] = A.state[(4 + k) * vstride + vbase + parent];
        }
        GgpFastConstsTable<N, TAB == 2> kp{SMEM ? ks : kv, F.dt_idx};
        bool valid = true;
        own = ggp_fast_cell<double, N>(F, slot, sp, s, kp, valid);
        if (F.s_d1[slot] >= 0 || F.s_d2[slot] >= 0) {
#pragma unroll
            for (int k = 0; k < 4; ++k) A.state[k * vstride + vbase + slot] = s.m[k];
#pragma unroll
            for (int k = 0; k < 10; ++k) A.state[(4 + k) * vstride + vbase + slot] = s.c[k];
        }
        if (A.cell_ll) A.cell_ll[(int64_t)(A.v0 + v) * F.n_cells + F.s_cell[slot]] = own;
        if (!valid) invalid[A.v0 + v] = 1;
    }
    // fixed-order reduction: xor-shuffle tree inside the warp, then the warps in index order
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) own = own + __shfl_xor_sync(0xffffffffu, own, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = own;
    __syncthreads();
    if (threadIdx.x == 0) {
        double bs = 0.0;
        for (int i = 0; i < GGP_FAST_BLOCK / 32; ++i) bs = bs + red[i];
        A.partial[(int64_t)v * A.n_partial + A.partial0 + blockIdx.x] = bs;
    }
}

bool ggp_fast_supported_nodes(int n) { return n == 4 || n == 5 || n == 6 || n == 8 || n == 10; }


#define GGP_FAST_DISPATCH(n_nodes, CALL)                    \
    switch (n_nodes) {                                      \
        case 4: { constexpr int NN = 4; CALL; } break;      \
        case 5: { constexpr int NN = 5; CALL; } break;      \
        case 6: { constexpr int NN = 6; CALL; } break;      \
        case 8: { constexpr int NN = 8; CALL; } break;      \
        case 10: { constexpr int NN = 10; CALL; } break;    \
        default: return cudaErrorInvalidValue;              \
    }

size_t ggp_fast_consts_bytes(int n_nodes) {
    switch (n_nodes) {
        case 4: return sizeof(GgpFastConsts<double, 4>);
        case 5: return sizeof(GgpFastConsts<double, 5>);
        case 6: return sizeof(GgpFastConsts<double, 6>);
        case 8: return sizeof(GgpFastConsts<double, 8>);
        case 10: return sizeof(GgpFastConsts<double, 10>);
    }
    return 0;
}

cudaError_t ggp_fast_consts_launch(const GgpFwdArgs& A, const double* dt_values, int n_dt, void* ktab, int n_nodes, cudaStream_t stream) {
    const unsigned grid = (unsigned)((n_dt * A.v_count + 127) / 128);
    GGP_FAST_DISPATCH(n_nodes, (ggp_fast_consts_kernel<NN><<<grid, 128, 0, stream>>>(A, dt_values, n_dt, static_cast<GgpFastConsts<double, NN>*>(ktab))))
    return cudaGetLastError();
}

cudaError_t ggp_fast_loglik_launch(const GgpDevForest& F, const GgpFwdArgs& A, const void* ktab, int* invalid, int n_nodes,
                                   cudaStream_t stream) {
    const dim3 grid((unsigned)((A.n_slots + GGP_FAST_BLOCK - 1) / GGP_FAST_BLOCK), (unsigned)A.v_count);
    const int tab = F.n_dt == 1 ? 2 : (F.n_dt <= GGP_FAST_SMEM_DT ? 1 : 0);
#define GGP_FAST_LAUNCH(TB) GGP_FAST_DISPATCH(n_nodes, (ggp_fast_loglik_kernel<NN, TB><<<grid, GGP_FAST_BLOCK, 0, stream>>>(F, A, static_cast<const GgpFastConsts<double, NN>*>(ktab), invalid)))
    if (tab == 2) {
        GGP_FAST_LAUNCH(2)
    } else if (tab == 1) {
        GGP_FAST_LAUNCH(1)
    } else {
        GGP_FAST_LAUNCH(0)
    }
#undef GGP_FAST_LAUNCH
    return cudaGetLastError();
}
