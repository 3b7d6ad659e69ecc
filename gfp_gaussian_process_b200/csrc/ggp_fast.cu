// ggp_fast.cu — the FAST likelihood kernels (ggp_fast.cuh): one thread per (cell, parameter vector), one launch per
// generation, mother -> daughter hand-over through the same SoA state buffer and the same fixed-order reduction as the strict
// path.  Compiled with FMA contraction ON (-fmad=true); nothing of the strict math is included here.
//
// What depends on (parameters, dt) only - exp(-b t), the OU noise terms, the quadrature nodes t xi_j and exp(-+gq t xi_j):
// 16 + 16 N doubles, pre-multiplied for the quadrature sums - is tabulated once per (vector, distinct dt of the forest) by ggp_fast_consts_kernel; the forest stores
// the table index of every time point (2 bytes per point instead of the 8-byte time stamp).  Tables of up to
// GGP_FAST_SMEM_DT entries are staged in shared memory, larger ones are read through L1.
//
// The gradient kernels at the end of the file run the same code over dual numbers (ggp_dual.cuh): value and derivatives of
// the log-likelihood along chosen parameter directions in one pass (forward mode).
//
// Build: nvcc -std=c++17 -O3 -fmad=true -gencode arch=compute_100a,code=sm_100a -lineinfo -c
#include "ggp_fast_api.h"
#include "ggp_fast.cuh"
#include "ggp_dual.cuh"

#define GGP_FAST_BLOCK 128
#define GGP_FAST_SMEM_DT 16
#define GGP_GRAD_SMEM_DT 8   // entries of the gradient kernel's shared table: 8 dual entries of 10 nodes are 22.5 kB

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

template <class T, int N, bool ONE>
struct GgpFastConstsTable {
    const GgpFastConsts<T, N>* tab;   // this vector's entries
    const uint16_t* __restrict__ idx;
    // ONE: the forest has a single distinct time step (a fixed acquisition interval): no index to read.  The zero comes out of
    // an opaque instruction: with a literal the compiler hoists the entry's 16 + 16 N loads out of the step loop (1.5 kB of spills)
    __device__ __forceinline__ const GgpFastConsts<T, N>& at(int64_t k, int64_t) const {
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
        GgpFastConstsTable<double, N, TAB == 2> kp{SMEM ? ks : kv, F.dt_idx};
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

// ---- the gradient: the same kernels over dual numbers (ggp_dual.cuh) ------------------------------------------------------
// A thread carries GGP_GRAD_D directions of one (cell, vector): grid.y runs over (vector, direction block) pairs, pair =
// v * n_blocks + b, and every pair is an independent evaluation with its own constants table, state rows and partial sums.
// One direction per thread: at 2 blocks per SM the dual step already needs 255 registers and spills (DESIGN.md 5.6); two
// directions per thread spilled 7 times as much in a compile probe.
typedef GgpDual<GGP_GRAD_D> GgpGradT;

// the parameters of pair (v, b) as dual numbers: tangent k of block b is d / d p[dirs.idx[b * D + k]] (zero past dirs.n)
__device__ __forceinline__ GgpGradT ggp_grad_param(const GgpFwdArgs& A, const GgpGradDirs& G, int v, int b, int i) {
    GgpGradT x(A.params[(int64_t)(A.v0 + v) * GGP_NP + i]);
#pragma unroll
    for (int k = 0; k < GGP_GRAD_D; ++k) {
        const int j = b * GGP_GRAD_D + k;
        x.d[k] = (j < G.n && G.idx[j] == i) ? 1.0 : 0.0;
    }
    return x;
}

template <int N>
__global__ void __launch_bounds__(128) ggp_fast_grad_consts_kernel(const GgpFwdArgs A, const GgpGradDirs G, const double* __restrict__ dt_values,
                                                                   int n_dt, GgpFastConsts<GgpGradT, N>* __restrict__ ktab) {
    const int nb = (G.n + GGP_GRAD_D - 1) / GGP_GRAD_D;
    const int i = blockIdx.x * 128 + threadIdx.x;
    if (i >= n_dt * A.v_count * nb) return;
    const int pair = i / n_dt, d = i - pair * n_dt;
    const int v = pair / nb, b = pair - v * nb;
    GgpGradT p[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) p[k] = ggp_grad_param(A, G, v, b, k);
    GgpFastConsts<GgpGradT, N> K;
    ggp_fast_consts(K, GgpGradT(dt_values[d]), p[0], p[1], p[2], p[3], p[4], p[5], p[6], GgpGLRule<N>());
    ktab[i] = K;
}

// one generation (or upload chunk of it) of the gradient; block (x, pair).  State rows: 14 x (1 + D), row r * (1 + D) + j
// holds component r (4 means, then the upper triangle) of the value (j = 0) or of tangent j - 1.  Partials: the value and
// every tangent in its own row (pair * (1 + D) + j), reduced in the likelihood's fixed order.
// TAB as ggp_fast_loglik_kernel; the shared copy holds up to GGP_GRAD_SMEM_DT entries (a dual entry is twice as large)
template <int N, int TAB>
__global__ void __launch_bounds__(GGP_FAST_BLOCK, 2) ggp_fast_grad_kernel(const GgpDevForest F, const GgpFwdArgs A, const GgpGradDirs G,
                                                                      const GgpFastConsts<GgpGradT, N>* __restrict__ ktab,
                                                                      int* __restrict__ invalid) {
    constexpr int C = 1 + GGP_GRAD_D;
    __shared__ GgpGradT sp[GGP_NP];
    __shared__ double red[C][GGP_FAST_BLOCK / 32];
    constexpr bool SMEM = TAB != 0;
    __shared__ GgpFastConsts<GgpGradT, N> ks[TAB == 1 ? GGP_GRAD_SMEM_DT : 1];
    const int nb = (G.n + GGP_GRAD_D - 1) / GGP_GRAD_D;
    const int lane_slot = blockIdx.x * GGP_FAST_BLOCK + threadIdx.x;
    const bool active = lane_slot < A.n_slots;
    const int slot = A.slot0 + (active ? lane_slot : 0);
    const int pair = blockIdx.y;
    const int v = pair / nb, b = pair - v * nb;
    if (threadIdx.x < GGP_NP) sp[threadIdx.x] = ggp_grad_param(A, G, v, b, threadIdx.x);
    const GgpFastConsts<GgpGradT, N>* kv = ktab + (int64_t)pair * F.n_dt;
    if (SMEM) {
        const double* src = reinterpret_cast<const double*>(kv);
        double* dst = reinterpret_cast<double*>(ks);
        for (int i = threadIdx.x; i < F.n_dt * (int)(sizeof(GgpFastConsts<GgpGradT, N>) / sizeof(double)); i += GGP_FAST_BLOCK) dst[i] = src[i];
    }
    __syncthreads();
    GgpGradT own(0.0);
    if (active) {
        const int64_t vstride = (int64_t)A.v_count * nb * F.n_cells;
        const int64_t vbase = (int64_t)pair * F.n_cells;
        const int parent = F.s_parent[slot];
        GgpFastState<GgpGradT> s;
        if (parent >= 0) {
#pragma unroll
            for (int k = 0; k < 14; ++k) {
                GgpGradT& x = k < 4 ? s.m[k] : s.c[k - 4];
                x.v = A.state[(k * C) * vstride + vbase + parent];
#pragma unroll
                for (int j = 0; j < GGP_GRAD_D; ++j) x.d[j] = A.state[(k * C + 1 + j) * vstride + vbase + parent];
            }
        }
        GgpFastConstsTable<GgpGradT, N, TAB == 2> kp{SMEM ? ks : kv, F.dt_idx};
        bool valid = true;
        own = ggp_fast_cell<GgpGradT, N>(F, slot, sp, s, kp, valid);
        if (F.s_d1[slot] >= 0 || F.s_d2[slot] >= 0) {
#pragma unroll
            for (int k = 0; k < 14; ++k) {
                const GgpGradT& x = k < 4 ? s.m[k] : s.c[k - 4];
                A.state[(k * C) * vstride + vbase + slot] = x.v;
#pragma unroll
                for (int j = 0; j < GGP_GRAD_D; ++j) A.state[(k * C + 1 + j) * vstride + vbase + slot] = x.d[j];
            }
        }
        if (!valid) invalid[A.v0 + v] = 1;
    }
    // fixed-order reduction of the value and of every tangent: xor-shuffle tree inside the warp, then the warps in index order
    double part[C];
    part[0] = own.v;
#pragma unroll
    for (int j = 0; j < GGP_GRAD_D; ++j) part[1 + j] = own.d[j];
#pragma unroll
    for (int c = 0; c < C; ++c) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) part[c] = part[c] + __shfl_xor_sync(0xffffffffu, part[c], o);
        if ((threadIdx.x & 31) == 0) red[c][threadIdx.x >> 5] = part[c];
    }
    __syncthreads();
    if (threadIdx.x < C) {
        double bs = 0.0;
        for (int i = 0; i < GGP_FAST_BLOCK / 32; ++i) bs = bs + red[threadIdx.x][i];
        A.partial[((int64_t)pair * C + threadIdx.x) * A.n_partial + A.partial0 + blockIdx.x] = bs;
    }
}

size_t ggp_fast_grad_consts_bytes(int n_nodes) {
    switch (n_nodes) {
        case 4: return sizeof(GgpFastConsts<GgpGradT, 4>);
        case 5: return sizeof(GgpFastConsts<GgpGradT, 5>);
        case 6: return sizeof(GgpFastConsts<GgpGradT, 6>);
        case 8: return sizeof(GgpFastConsts<GgpGradT, 8>);
        case 10: return sizeof(GgpFastConsts<GgpGradT, 10>);
    }
    return 0;
}

cudaError_t ggp_fast_grad_consts_launch(const GgpFwdArgs& A, const GgpGradDirs& G, const double* dt_values, int n_dt, void* ktab,
                                        int n_nodes, cudaStream_t stream) {
    const int nb = (G.n + GGP_GRAD_D - 1) / GGP_GRAD_D;
    const unsigned grid = (unsigned)(((int64_t)n_dt * A.v_count * nb + 127) / 128);
    GGP_FAST_DISPATCH(n_nodes, (ggp_fast_grad_consts_kernel<NN><<<grid, 128, 0, stream>>>(A, G, dt_values, n_dt, static_cast<GgpFastConsts<GgpGradT, NN>*>(ktab))))
    return cudaGetLastError();
}

cudaError_t ggp_fast_grad_launch(const GgpDevForest& F, const GgpFwdArgs& A, const GgpGradDirs& G, const void* ktab, int* invalid,
                                 int n_nodes, cudaStream_t stream) {
    const int nb = (G.n + GGP_GRAD_D - 1) / GGP_GRAD_D;
    const dim3 grid((unsigned)((A.n_slots + GGP_FAST_BLOCK - 1) / GGP_FAST_BLOCK), (unsigned)(A.v_count * nb));
    const int tab = F.n_dt == 1 ? 2 : (F.n_dt <= GGP_GRAD_SMEM_DT ? 1 : 0);
#define GGP_GRAD_LAUNCH(TB) GGP_FAST_DISPATCH(n_nodes, (ggp_fast_grad_kernel<NN, TB><<<grid, GGP_FAST_BLOCK, 0, stream>>>(F, A, G, static_cast<const GgpFastConsts<GgpGradT, NN>*>(ktab), invalid)))
    if (tab == 2) {
        GGP_GRAD_LAUNCH(2)
    } else if (tab == 1) {
        GGP_GRAD_LAUNCH(1)
    } else {
        GGP_GRAD_LAUNCH(0)
    }
#undef GGP_GRAD_LAUNCH
    return cudaGetLastError();
}
