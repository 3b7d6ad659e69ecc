// ggp_fast.cu — the FAST likelihood kernels (ggp_fast.cuh): one thread per (cell, parameter vector), one launch per
// generation, mother -> daughter hand-over through the same SoA state buffer and the same fixed-order reduction as the strict
// path.  Compiled with FMA contraction ON (-fmad=true); nothing of the strict math is included here.
//
// What depends on (parameters, dt) only - exp(-b t), the OU noise terms, the quadrature nodes t xi_j and exp(-+gq t xi_j):
// 16 + 16 N doubles, pre-multiplied for the quadrature sums - is tabulated once per (vector, distinct dt of the forest) by ggp_fast_consts_kernel; the forest stores
// the table index of every time point (2 bytes per point instead of the 8-byte time stamp).  Tables of up to
// GGP_FAST_SMEM_DT entries are staged in shared memory, larger ones are read through L1.
//
// The derivative kernels at the end of the file run the same code over dual numbers and second-order Taylor numbers
// (ggp_dual.cuh): value, derivatives and second derivatives of the log-likelihood along chosen parameter directions in one
// pass (forward mode).
//
// Build: nvcc -std=c++17 -O3 -fmad=true -gencode arch=compute_100a,code=sm_100a -lineinfo -c
#include "ggp_fast_api.h"
#include "ggp_fast.cuh"
#include "ggp_dual.cuh"

#define GGP_FAST_BLOCK 128
#define GGP_FAST_SMEM_DT 16
#define GGP_GRAD_SMEM_DT 8   // entries of the gradient kernel's shared table: 8 dual entries of 10 nodes are 22.5 kB
#define GGP_HESS_SMEM_DT 5   // entries of the Hessian kernel's shared table: 5 GgpTaylor2 entries of 10 nodes are 21.1 kB

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

// ---- derivatives: the same kernels over dual numbers and second-order Taylor numbers (ggp_dual.cuh) -------------------------
// Every vector is evaluated several times, each evaluation along its own seeding of the parameters: grid.y runs over (vector,
// evaluation) pairs, pair = v * n_evals + e, and every pair is an independent evaluation with its own constants table, state
// rows and partial sums.  A seeding S names the scalar and how evaluation e seeds parameter i:
//   GgpGradSeed  GgpDual<GGP_GRAD_D>: evaluation b is direction block b, tangent k = d / d p[G.idx[b * D + k]];
//   GgpHessSeed  GgpTaylor2: evaluation e steps along u = s_a e_a + s_b e_b (a = H.a[e], b = H.b[e], s = ggp_hess_scale(p),
//                once if a == b) and returns (value, g.u, u^T H u).
// One direction per thread: at 2 blocks per SM the dual step already needs 255 registers and spills (DESIGN.md 5.6); two
// directions per thread spilled 7 times as much in a compile probe.
typedef GgpDual<GGP_GRAD_D> GgpGradT;

// the derivative parts of a scalar (C - 1 of them, after the value v)
template <int D>
__device__ __forceinline__ double& ggp_tan(GgpDual<D>& x, int j) { return x.d[j]; }
template <int D>
__device__ __forceinline__ const double& ggp_tan(const GgpDual<D>& x, int j) { return x.d[j]; }
__device__ __forceinline__ double& ggp_tan(GgpTaylor2& x, int j) { return j == 0 ? x.d : x.dd; }
__device__ __forceinline__ const double& ggp_tan(const GgpTaylor2& x, int j) { return j == 0 ? x.d : x.dd; }

struct GgpGradSeed {
    typedef GgpGradT T;
    typedef GgpGradDirs Dirs;
    static constexpr int C = 1 + GGP_GRAD_D;        // results per evaluation
    static constexpr int SMEM_DT = GGP_GRAD_SMEM_DT;
    static __host__ __device__ __forceinline__ int evals(const Dirs& G) { return (G.n + GGP_GRAD_D - 1) / GGP_GRAD_D; }
    // the parameters of pair (v, b) as dual numbers: tangent k of block b is d / d p[dirs.idx[b * D + k]] (zero past dirs.n)
    static __device__ __forceinline__ T param(const GgpFwdArgs& A, const Dirs& G, int v, int b, int i) {
        T x(A.params[(int64_t)(A.v0 + v) * GGP_NP + i]);
#pragma unroll
        for (int k = 0; k < GGP_GRAD_D; ++k) {
            const int j = b * GGP_GRAD_D + k;
            x.d[k] = (j < G.n && G.idx[j] == i) ? 1.0 : 0.0;
        }
        return x;
    }
};

struct GgpHessSeed {
    typedef GgpTaylor2 T;
    typedef GgpHessDirs Dirs;
    static constexpr int C = 3;
    static constexpr int SMEM_DT = GGP_HESS_SMEM_DT;
    static __host__ __device__ __forceinline__ int evals(const Dirs& H) { return H.n; }
    static __device__ __forceinline__ T param(const GgpFwdArgs& A, const Dirs& H, int v, int e, int i) {
        const double p = A.params[(int64_t)(A.v0 + v) * GGP_NP + i];
        return T(p, (H.a[e] == i || H.b[e] == i) ? ggp_hess_scale(p) : 0.0, 0.0);
    }
};

template <class S, int N>
__global__ void __launch_bounds__(128) ggp_fast_grad_consts_kernel(const GgpFwdArgs A, const typename S::Dirs G,
                                                                   const double* __restrict__ dt_values, int n_dt,
                                                                   GgpFastConsts<typename S::T, N>* __restrict__ ktab) {
    typedef typename S::T T;
    const int nb = S::evals(G);
    const int i = blockIdx.x * 128 + threadIdx.x;
    if (i >= n_dt * A.v_count * nb) return;
    const int pair = i / n_dt, d = i - pair * n_dt;
    const int v = pair / nb, b = pair - v * nb;
    T p[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) p[k] = S::param(A, G, v, b, k);
    GgpFastConsts<T, N> K;
    ggp_fast_consts(K, T(dt_values[d]), p[0], p[1], p[2], p[3], p[4], p[5], p[6], GgpGLRule<N>());
    ktab[i] = K;
}

// one generation (or upload chunk of it) of the derivatives; block (x, pair).  State rows: 14 x C, row r * C + j holds
// component r (4 means, then the upper triangle) of the value (j = 0) or of derivative part j - 1.  Partials: the value and
// every derivative part in its own row (pair * C + j), reduced in the likelihood's fixed order.
// TAB as ggp_fast_loglik_kernel; the shared copy holds up to S::SMEM_DT entries
template <class S, int N, int TAB>
__global__ void __launch_bounds__(GGP_FAST_BLOCK, 2) ggp_fast_grad_kernel(const GgpDevForest F, const GgpFwdArgs A, const typename S::Dirs G,
                                                                      const GgpFastConsts<typename S::T, N>* __restrict__ ktab,
                                                                      int* __restrict__ invalid) {
    typedef typename S::T T;
    constexpr int C = S::C;
    __shared__ T sp[GGP_NP];
    __shared__ double red[C][GGP_FAST_BLOCK / 32];
    constexpr bool SMEM = TAB != 0;
    __shared__ GgpFastConsts<T, N> ks[TAB == 1 ? S::SMEM_DT : 1];
    const int nb = S::evals(G);
    const int lane_slot = blockIdx.x * GGP_FAST_BLOCK + threadIdx.x;
    const bool active = lane_slot < A.n_slots;
    const int slot = A.slot0 + (active ? lane_slot : 0);
    const int pair = blockIdx.y;
    const int v = pair / nb, b = pair - v * nb;
    if (threadIdx.x < GGP_NP) sp[threadIdx.x] = S::param(A, G, v, b, threadIdx.x);
    const GgpFastConsts<T, N>* kv = ktab + (int64_t)pair * F.n_dt;
    if (SMEM) {
        const double* src = reinterpret_cast<const double*>(kv);
        double* dst = reinterpret_cast<double*>(ks);
        for (int i = threadIdx.x; i < F.n_dt * (int)(sizeof(GgpFastConsts<T, N>) / sizeof(double)); i += GGP_FAST_BLOCK) dst[i] = src[i];
    }
    __syncthreads();
    T own(0.0);
    if (active) {
        const int64_t vstride = (int64_t)A.v_count * nb * F.n_cells;
        const int64_t vbase = (int64_t)pair * F.n_cells;
        const int parent = F.s_parent[slot];
        GgpFastState<T> s;
        if (parent >= 0) {
#pragma unroll
            for (int k = 0; k < 14; ++k) {
                T& x = k < 4 ? s.m[k] : s.c[k - 4];
                x.v = A.state[(k * C) * vstride + vbase + parent];
#pragma unroll
                for (int j = 0; j < C - 1; ++j) ggp_tan(x, j) = A.state[(k * C + 1 + j) * vstride + vbase + parent];
            }
        }
        GgpFastConstsTable<T, N, TAB == 2> kp{SMEM ? ks : kv, F.dt_idx};
        bool valid = true;
        own = ggp_fast_cell<T, N>(F, slot, sp, s, kp, valid);
        if (F.s_d1[slot] >= 0 || F.s_d2[slot] >= 0) {
#pragma unroll
            for (int k = 0; k < 14; ++k) {
                const T& x = k < 4 ? s.m[k] : s.c[k - 4];
                A.state[(k * C) * vstride + vbase + slot] = x.v;
#pragma unroll
                for (int j = 0; j < C - 1; ++j) A.state[(k * C + 1 + j) * vstride + vbase + slot] = ggp_tan(x, j);
            }
        }
        if (!valid) invalid[A.v0 + v] = 1;
    }
    // fixed-order reduction of the value and of every derivative part: xor-shuffle tree inside the warp, then the warps in index order
    double part[C];
    part[0] = own.v;
#pragma unroll
    for (int j = 0; j < C - 1; ++j) part[1 + j] = ggp_tan(own, j);
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

namespace {

template <class T>
size_t consts_bytes(int n_nodes) {
    switch (n_nodes) {
        case 4: return sizeof(GgpFastConsts<T, 4>);
        case 5: return sizeof(GgpFastConsts<T, 5>);
        case 6: return sizeof(GgpFastConsts<T, 6>);
        case 8: return sizeof(GgpFastConsts<T, 8>);
        case 10: return sizeof(GgpFastConsts<T, 10>);
    }
    return 0;
}

template <class S>
cudaError_t derivs_consts_launch(const GgpFwdArgs& A, const typename S::Dirs& G, const double* dt_values, int n_dt, void* ktab,
                                 int n_nodes, cudaStream_t stream) {
    const unsigned grid = (unsigned)(((int64_t)n_dt * A.v_count * S::evals(G) + 127) / 128);
    GGP_FAST_DISPATCH(n_nodes, (ggp_fast_grad_consts_kernel<S, NN><<<grid, 128, 0, stream>>>(A, G, dt_values, n_dt, static_cast<GgpFastConsts<typename S::T, NN>*>(ktab))))
    return cudaGetLastError();
}

template <class S>
cudaError_t derivs_launch(const GgpDevForest& F, const GgpFwdArgs& A, const typename S::Dirs& G, const void* ktab, int* invalid,
                          int n_nodes, cudaStream_t stream) {
    const dim3 grid((unsigned)((A.n_slots + GGP_FAST_BLOCK - 1) / GGP_FAST_BLOCK), (unsigned)(A.v_count * S::evals(G)));
    const int tab = F.n_dt == 1 ? 2 : (F.n_dt <= S::SMEM_DT ? 1 : 0);
#define GGP_DERIVS_LAUNCH(TB) GGP_FAST_DISPATCH(n_nodes, (ggp_fast_grad_kernel<S, NN, TB><<<grid, GGP_FAST_BLOCK, 0, stream>>>(F, A, G, static_cast<const GgpFastConsts<typename S::T, NN>*>(ktab), invalid)))
    if (tab == 2) {
        GGP_DERIVS_LAUNCH(2)
    } else if (tab == 1) {
        GGP_DERIVS_LAUNCH(1)
    } else {
        GGP_DERIVS_LAUNCH(0)
    }
#undef GGP_DERIVS_LAUNCH
    return cudaGetLastError();
}

}  // namespace

size_t ggp_fast_grad_consts_bytes(int n_nodes) { return consts_bytes<GgpGradT>(n_nodes); }
size_t ggp_fast_hess_consts_bytes(int n_nodes) { return consts_bytes<GgpTaylor2>(n_nodes); }

cudaError_t ggp_fast_grad_consts_launch(const GgpFwdArgs& A, const GgpGradDirs& G, const double* dt_values, int n_dt, void* ktab,
                                        int n_nodes, cudaStream_t stream) {
    return derivs_consts_launch<GgpGradSeed>(A, G, dt_values, n_dt, ktab, n_nodes, stream);
}
cudaError_t ggp_fast_hess_consts_launch(const GgpFwdArgs& A, const GgpHessDirs& H, const double* dt_values, int n_dt, void* ktab,
                                        int n_nodes, cudaStream_t stream) {
    return derivs_consts_launch<GgpHessSeed>(A, H, dt_values, n_dt, ktab, n_nodes, stream);
}

cudaError_t ggp_fast_grad_launch(const GgpDevForest& F, const GgpFwdArgs& A, const GgpGradDirs& G, const void* ktab, int* invalid,
                                 int n_nodes, cudaStream_t stream) {
    return derivs_launch<GgpGradSeed>(F, A, G, ktab, invalid, n_nodes, stream);
}
cudaError_t ggp_fast_hess_launch(const GgpDevForest& F, const GgpFwdArgs& A, const GgpHessDirs& H, const void* ktab, int* invalid,
                                 int n_nodes, cudaStream_t stream) {
    return derivs_launch<GgpHessSeed>(F, A, H, ktab, invalid, n_nodes, stream);
}
