// ggp_fast.cu — the FAST likelihood kernels (ggp_fast.cuh): one thread per (cell, parameter vector, evaluation), one launch
// per generation, mother -> daughter hand-over through the same SoA state buffer and the same fixed-order reduction as the
// strict path.  Compiled with FMA contraction ON (-fmad=true); nothing of the strict math is included here.
//
// What depends on (parameters, dt) only - exp(-b t), the OU noise terms, the quadrature nodes t xi_j and exp(-+gq t xi_j):
// 10 + 20 N scalars, pre-multiplied for the quadrature sums - is tabulated once per (vector, evaluation, distinct dt of the
// forest) by ggp_fast_consts_kernel; the forest stores the table index of every time point (2 bytes per point instead of the
// 8-byte time stamp).  Small tables are staged in shared memory, larger ones are read through L1.
//
// One kernel pair serves the log-likelihood and its derivatives: a seeding picks the scalar - double, dual numbers or
// second-order Taylor numbers (ggp_dual.cuh) - and how each evaluation of a vector (GgpEvalPlan, ggp_types.cuh) seeds the
// parameters: value, derivatives and second derivatives along chosen parameter directions in one pass (forward mode).
//
// Build: nvcc -std=c++17 -O3 -fmad=true -gencode arch=compute_100a,code=sm_100a -lineinfo -c
#include "ggp_fast_api.h"
#include "ggp_fast.cuh"
#include "ggp_dual.cuh"

#include <type_traits>

#define GGP_FAST_BLOCK 128

// A seeding S says what one family instance of the kernels evaluates: the scalar T, the results per evaluation C (the
// components of T), the evaluations per vector (evals), the resident blocks per SM the registers are allocated for
// (MIN_BLOCKS), the entries of the shared constants table (SMEM_DT), how evaluation e seeds parameter i (param), whether
// the per-cell log-likelihood is written (CELL_LL: [n_vec][n_cells]) and whether every component of every cell is (CELL_ROWS:
// [pair][C][n_cells] of the launch, the per-tree scores' input).  Both go to A.cell_ll when it is not null.  grid.y runs over
// (vector, evaluation) pairs, pair = v * evals + e; every pair is an independent evaluation with its own constants table, state
// rows and partial sums.
//   GgpValueSeed  double: the log-likelihood, device or inline parameters.  3 blocks per SM: 2 / 3 / 4 blocks (242 / 168 / 128
//                 registers) measured 0.777 / 0.752 / 0.864 ms on configs[1] with 6 nodes; 16 table entries.
//   GgpGradSeed   GgpDual<1>: evaluation e is direction P.a[e], results (value, g.e_a).  One direction per thread: at 2 blocks per
//                 SM the dual step already needs 255 registers and spills (DESIGN.md 5.6), two per thread spilled 7 times as much
//                 in a compile probe.  8 dual entries of 10 nodes are 26.9 kB.
//   GgpHessSeed   GgpTaylor2: evaluation e steps along u = s_a e_a + s_b e_b (a = P.a[e], b = P.b[e], s = ggp_hess_scale(p), once
//                 if a == b) and returns (value, g.u, u^T H u).  5 entries of 10 nodes are 25.2 kB.
// The derivative seedings read device parameters.
struct GgpValueSeed {
    typedef double T;
    static constexpr int C = 1, MIN_BLOCKS = 3, SMEM_DT = 16;
    static constexpr bool CELL_LL = true, CELL_ROWS = false;
    static __device__ __forceinline__ int evals(const GgpEvalPlan&) { return 1; }
    static __device__ __forceinline__ T param(const GgpFwdArgs& A, const GgpEvalPlan&, int v, int, int i) {
        return A.params ? A.params[(int64_t)(A.v0 + v) * GGP_NP + i] : A.inline_params[(A.v0 + v) * GGP_NP + i];
    }
};

struct GgpGradSeed {
    typedef GgpDual<1> T;
    static constexpr int C = 2, MIN_BLOCKS = 2, SMEM_DT = 8;
    static constexpr bool CELL_LL = false, CELL_ROWS = true;
    static __device__ __forceinline__ int evals(const GgpEvalPlan& P) { return P.n_run; }
    static __device__ __forceinline__ T param(const GgpFwdArgs& A, const GgpEvalPlan& P, int v, int e, int i) {
        T x(A.params[(int64_t)(A.v0 + v) * GGP_NP + i]);
        x.d[0] = P.seeds(e, i) ? 1.0 : 0.0;
        return x;
    }
};

struct GgpHessSeed {
    typedef GgpTaylor2 T;
    static constexpr int C = 3, MIN_BLOCKS = 2, SMEM_DT = 5;
    static constexpr bool CELL_LL = false, CELL_ROWS = false;
    static __device__ __forceinline__ int evals(const GgpEvalPlan& P) { return P.n_run; }
    static __device__ __forceinline__ T param(const GgpFwdArgs& A, const GgpEvalPlan& P, int v, int e, int i) {
        const double p = A.params[(int64_t)(A.v0 + v) * GGP_NP + i];
        return T(p, P.seeds(e, i) ? ggp_hess_scale(p) : 0.0, 0.0);
    }
};

// the (parameters, dt)-only constants of every (pair, distinct time step): ktab[pair * n_dt + d].  One thread per node of an
// entry and one for the rest of it: the nodes are independent, and an entry in one thread spilled (dual and Taylor scalars)
template <class S, int N>
__global__ void __launch_bounds__(128) ggp_fast_consts_kernel(const GgpFwdArgs A, const double* __restrict__ dt_values, int n_dt,
                                                              GgpFastConsts<typename S::T, N>* __restrict__ ktab, const GgpEvalPlan P) {
    typedef typename S::T T;
    const int ne = S::evals(P);
    const int i = blockIdx.x * 128 + threadIdx.x;
    const int entry = i / (N + 1), j = i - entry * (N + 1);   // j < N: node j, j == N: the rest
    if (entry >= n_dt * A.v_count * ne) return;
    const int pair = entry / n_dt, d = entry - pair * n_dt;
    const int v = pair / ne, e = pair - v * ne;
    const T t = T(dt_values[d]);
    GgpFastConsts<T, N>& K = ktab[entry];
    if (j < N) {
        ggp_fast_consts_node(K.node[j], j, t, S::param(A, P, v, e, 3), S::param(A, P, v, e, 4), S::param(A, P, v, e, 5), GgpGLRule<N>());
    } else {
        ggp_fast_consts_head(K, t, S::param(A, P, v, e, 1), S::param(A, P, v, e, 2), S::param(A, P, v, e, 4), S::param(A, P, v, e, 5),
                             S::param(A, P, v, e, 6));
    }
}

template <class T, int N, bool ONE>
struct GgpFastConstsTable {
    const GgpFastConsts<T, N>* tab;   // this vector's entries
    const uint16_t* __restrict__ idx;
    // ONE: the forest has a single distinct time step (a fixed acquisition interval): no index to read.  The zero comes out of
    // an opaque instruction: with a literal the compiler hoists the entry's loads out of the step loop (1.5 kB of spills)
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

// one generation (or upload chunk of it); block (x, pair).  State rows: 14 x C, row r * C + j holds component j (ggp_comp) of
// state component r (4 means, then the upper triangle).  Partials: every component in its own row (pair * C + j), reduced in a
// fixed order.  invalid [n_vec]: set for a vector whose evaluation left the rule's validity range or met a NaN term.
// TAB 0: the constants table is read through L1; 1: it fits the block's shared copy (n_dt <= S::SMEM_DT): shared-memory loads
// with known address space; 2: one entry (n_dt == 1), shared, and the per-point index is not read at all (its load was the
// kernel's one exposed memory latency: the table address of a step depends on it)
template <class S, int N, int TAB>
__global__ void __launch_bounds__(GGP_FAST_BLOCK, S::MIN_BLOCKS) ggp_fast_loglik_kernel(const GgpDevForest F, const GgpFwdArgs A,
                                                                                    const GgpFastConsts<typename S::T, N>* __restrict__ ktab,
                                                                                    int* __restrict__ invalid, const GgpEvalPlan P) {
    typedef typename S::T T;
    constexpr int C = S::C;
    __shared__ T sp[GGP_NP];
    __shared__ double red[C][GGP_FAST_BLOCK / 32];
    constexpr bool SMEM = TAB != 0;
    __shared__ GgpFastConsts<T, N> ks[TAB == 1 ? S::SMEM_DT : 1];
    const int ne = S::evals(P);
    const int lane_slot = blockIdx.x * GGP_FAST_BLOCK + threadIdx.x;
    const bool active = lane_slot < A.n_slots;
    const int slot = A.slot0 + (active ? lane_slot : 0);
    const int pair = blockIdx.y;
    const int v = pair / ne, e = pair - v * ne;
    if (threadIdx.x < GGP_NP) sp[threadIdx.x] = S::param(A, P, v, e, threadIdx.x);
    const GgpFastConsts<T, N>* kv = ktab + (int64_t)pair * F.n_dt;
    if (SMEM) {
        const double* src = reinterpret_cast<const double*>(kv);
        double* dst = reinterpret_cast<double*>(ks);
        for (int i = threadIdx.x; i < F.n_dt * (int)(sizeof(GgpFastConsts<T, N>) / sizeof(double)); i += GGP_FAST_BLOCK) dst[i] = src[i];
    }
    __syncthreads();
    T own(0.0);
    if (active) {
        const int64_t vstride = (int64_t)A.v_count * ne * F.n_cells;
        const int64_t vbase = (int64_t)pair * F.n_cells;
        const int parent = F.s_parent[slot];
        GgpFastState<T> s;
        if (parent >= 0) {
#pragma unroll
            for (int k = 0; k < 14; ++k) {
                T& x = k < 4 ? s.m[k] : s.c[k - 4];
#pragma unroll
                for (int j = 0; j < C; ++j) ggp_comp(x, j) = A.state[(k * C + j) * vstride + vbase + parent];
            }
        }
        GgpFastConstsTable<T, N, TAB == 2> kp{SMEM ? ks : kv, F.dt_idx};
        bool valid = true;
        own = ggp_fast_cell<T, N>(F, slot, sp, s, kp, valid);
        if (F.s_d1[slot] >= 0 || F.s_d2[slot] >= 0) {
#pragma unroll
            for (int k = 0; k < 14; ++k) {
                T& x = k < 4 ? s.m[k] : s.c[k - 4];
#pragma unroll
                for (int j = 0; j < C; ++j) A.state[(k * C + j) * vstride + vbase + slot] = ggp_comp(x, j);
            }
        }
        if (S::CELL_LL && A.cell_ll) A.cell_ll[(int64_t)(A.v0 + v) * F.n_cells + F.s_cell[slot]] = ggp_comp(own, 0);
        if (S::CELL_ROWS && A.cell_ll) {
#pragma unroll
            for (int j = 0; j < C; ++j) A.cell_ll[((int64_t)pair * C + j) * F.n_cells + F.s_cell[slot]] = ggp_comp(own, j);
        }
        if (!valid) invalid[A.v0 + v] = 1;
    }
    // fixed-order reduction of every component: xor-shuffle tree inside the warp, then the warps in index order
    double part[C];
#pragma unroll
    for (int c = 0; c < C; ++c) {
        part[c] = ggp_comp(own, c);
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

// per-tree sums of per-cell rows: one warp per (row, tree).  The lanes stride over the tree's cells in the order tree_cells
// lists them, then an xor-shuffle tree: the sum depends on the tree's cell list only, not on the grid
__global__ void __launch_bounds__(256) ggp_tree_sum_kernel(const double* __restrict__ rows, int64_t n_cells, int64_t n_rows,
                                                           const int64_t* __restrict__ tree_off, const int32_t* __restrict__ tree_cells,
                                                           int32_t n_trees, double* __restrict__ out) {
    const int64_t w = ((int64_t)blockIdx.x * 256 + threadIdx.x) >> 5;   // warp-uniform: whole warps leave together
    const int lane = threadIdx.x & 31;
    if (w >= n_rows * n_trees) return;
    const int64_t r = w / n_trees, t = w - r * n_trees;
    const double* row = rows + r * n_cells;
    double s = 0.0;
    for (int64_t i = tree_off[t] + lane; i < tree_off[t + 1]; i += 32) s = s + row[tree_cells[i]];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s = s + __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) out[r * n_trees + t] = s;
}

bool ggp_fast_supported_nodes(int n) { return n == 4 || n == 5 || n == 6 || n == 8 || n == 10; }

namespace {

// f(S(), std::integral_constant<int, N>()) with the rule of n_nodes; false for an unsupported rule
template <class S, class Fn>
bool with_nodes(int n_nodes, Fn&& f) {
    switch (n_nodes) {
        case 4: f(S(), std::integral_constant<int, 4>()); return true;
        case 5: f(S(), std::integral_constant<int, 5>()); return true;
        case 6: f(S(), std::integral_constant<int, 6>()); return true;
        case 8: f(S(), std::integral_constant<int, 8>()); return true;
        case 10: f(S(), std::integral_constant<int, 10>()); return true;
    }
    return false;
}

// with_nodes with the seeding of the plan's order
template <class Fn>
bool with_seed(const GgpEvalPlan& P, int n_nodes, Fn&& f) {
    if (P.order == 2) return with_nodes<GgpHessSeed>(n_nodes, f);
    if (P.order == 1) return with_nodes<GgpGradSeed>(n_nodes, f);
    return with_nodes<GgpValueSeed>(n_nodes, f);
}

}  // namespace

size_t ggp_fast_consts_bytes(const GgpEvalPlan& P, int n_nodes) {
    size_t bytes = 0;
    with_seed(P, n_nodes, [&](auto s, auto n) { bytes = sizeof(GgpFastConsts<typename decltype(s)::T, decltype(n)::value>); });
    return bytes;
}

cudaError_t ggp_fast_consts_launch(const GgpFwdArgs& A, const GgpEvalPlan& P, const double* dt_values, int n_dt, void* ktab, int n_nodes,
                                   cudaStream_t stream) {
    const bool ok = with_seed(P, n_nodes, [&](auto s, auto n) {
        typedef decltype(s) S;
        constexpr int N = decltype(n)::value;
        const unsigned grid = (unsigned)(((int64_t)n_dt * A.v_count * P.n_run * (N + 1) + 127) / 128);
        ggp_fast_consts_kernel<S, N><<<grid, 128, 0, stream>>>(A, dt_values, n_dt, static_cast<GgpFastConsts<typename S::T, N>*>(ktab), P);
    });
    return ok ? cudaGetLastError() : cudaErrorInvalidValue;
}

cudaError_t ggp_tree_sum_launch(const double* rows, int64_t n_cells, int64_t n_rows, const int64_t* tree_off, const int32_t* tree_cells,
                                int32_t n_trees, double* out, cudaStream_t stream) {
    const int64_t warps = n_rows * n_trees;
    if (warps == 0) return cudaSuccess;
    ggp_tree_sum_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, stream>>>(rows, n_cells, n_rows, tree_off, tree_cells, n_trees, out);
    return cudaGetLastError();
}

cudaError_t ggp_fast_loglik_launch(const GgpDevForest& F, const GgpFwdArgs& A, const GgpEvalPlan& P, const void* ktab, int* invalid,
                                   int n_nodes, cudaStream_t stream) {
    const dim3 grid((unsigned)((A.n_slots + GGP_FAST_BLOCK - 1) / GGP_FAST_BLOCK), (unsigned)(A.v_count * P.n_run));
    const bool ok = with_seed(P, n_nodes, [&](auto s, auto n) {
        typedef decltype(s) S;
        constexpr int N = decltype(n)::value;
        const auto* k = static_cast<const GgpFastConsts<typename S::T, N>*>(ktab);
        if (F.n_dt == 1)
            ggp_fast_loglik_kernel<S, N, 2><<<grid, GGP_FAST_BLOCK, 0, stream>>>(F, A, k, invalid, P);
        else if (F.n_dt <= S::SMEM_DT)
            ggp_fast_loglik_kernel<S, N, 1><<<grid, GGP_FAST_BLOCK, 0, stream>>>(F, A, k, invalid, P);
        else
            ggp_fast_loglik_kernel<S, N, 0><<<grid, GGP_FAST_BLOCK, 0, stream>>>(F, A, k, invalid, P);
    });
    return ok ? cudaGetLastError() : cudaErrorInvalidValue;
}
