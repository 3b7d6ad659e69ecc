// ggp_sim.cuh — measurement series simulated from the model on the forest's own genealogy, time grid and segments
// (ggp_simulate): the process synthetic.py defines, one thread per cell, one launch per generation.
//
// Per cell, with p = params[segment] of the point named:
//   root      x ~ N(m_x, v_x), g ~ N(m_g, v_g) (the root prior), lambda, q from their stationary OU laws (first point's p);
//   interval  `substeps` equal sub-intervals h of dt, p of the point the interval starts from; per sub-interval, in this order:
//             g += (e^x q - beta g) h; x += lambda h; lambda and q take exact OU transitions over h;
//   point     x_obs = x + N(0, var_x); g_obs = g + N(0, var_g) (const) or N(0, var_g max(g + fp_auto, 0)) (scaled);
//   division  the mother integrates from her last point to her daughters' first time (the earlier one if they differ) and
//             both daughters start from that state; the later daughter integrates the rest.  Then, with the mother's
//             last-point p: x -> x - log 2 + N(0, var_dx); g -> g / 2 + N(0, var_dg) (gauss) or
//             var_dg * Binomial(max(rint(g / var_dg), 1), 1/2) (binomial); lambda and q are inherited.
//
// Random numbers: Philox4x32-10 (Salmon et al., SC'11, "Parallel random numbers: as easy as 1, 2, 3"), key = the 64-bit seed,
// counter = (c0, c1, c2, c3):
//   c0  the cell's index in the caller's cell order (a group shard uses the caller's index, not its own)
//   c1  point index t: the observation at point t, the interval that starts there (t = n - 1: the gap to the daughters);
//       0xffffffff: a daughter's own work before her first point (the rest of the gap, the division)
//   c2  sub-interval index (OU draws); the high bits of the block index (binomial bits); else 0
//   c3  purpose << 24 | attempt (normals: the polar method's attempt; binomial bits: the low 24 bits of the block index)
// so the bits depend on the seed and the caller's indices only, not on the launch shape, the slot order or the sharding.
// Normals: Marsaglia's polar method on two 53-bit uniforms per Philox call (two normals per accepted call); it needs only
// ggp_log, sqrt and division, so the host build (g++ -ffp-contract=off) returns the device's bits.
// Binomial(n, 1/2): the popcount of n fair bits of the counter stream, exact; the cost is linear in n (about 43 000 bits, 340
// Philox calls, per division for the example data set's parameters: mq / (ml + beta) / var_dg).  n above 2^32 gives NaN.
#pragma once
#include <stdint.h>

#include "ggp_types.cuh"
#include "ggp_libm.cuh"

enum { GGP_SIM_ROOT_XG = 1, GGP_SIM_ROOT_LQ = 2, GGP_SIM_OU = 3, GGP_SIM_OBS = 4, GGP_SIM_DIV = 5, GGP_SIM_BITS = 6 };
#define GGP_SIM_BEFORE_FIRST 0xffffffffu
#define GGP_SIM_BLOCK 128

struct GgpSimArgs {
    int slot0, n_slots;            // this generation
    const double* params;          // [n_seg][11]
    double root[4];                // root prior m_x, m_g, v_x, v_g
    uint64_t seed;
    int substeps;
    const int64_t* key;            // NULL: c0 = the handle's cell index; else key[that index] (a group shard: the caller's)
    double* end;                   // [4][n_cells] by slot: x, g, lambda, q of a mother at her daughters' first time
    double* edge;                  // [4][n_cells] by the handle's cell: first x_obs, last x_obs, first g_obs, last g_obs
    unsigned long long* bad_key;   // min c0 of a cell with a non-finite observation
    double* x_out;                 // [n_ctp] the handle's log_length, caller's order
    double* g_out;                 // [n_ctp] the handle's fp
};

GGP_HD void ggp_mulhilo32(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
#if defined(__CUDA_ARCH__)
    hi = __umulhi(a, b);
    lo = a * b;
#else
    const uint64_t p = (uint64_t)a * b;
    hi = (uint32_t)(p >> 32);
    lo = (uint32_t)p;
#endif
}

// Philox4x32-10: ten rounds of c = (hi(M1 c2) ^ c1 ^ k0, lo(M1 c2), hi(M0 c0) ^ c3 ^ k1, lo(M0 c0)), the key bumped by the Weyl
// constants between rounds
GGP_HD void ggp_philox4x32_10(const uint32_t ctr[4], uint64_t key, uint32_t out[4]) {
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3];
    uint32_t k0 = (uint32_t)key, k1 = (uint32_t)(key >> 32);
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0, lo0, hi1, lo1;
        ggp_mulhilo32(0xD2511F53u, c0, hi0, lo0);
        ggp_mulhilo32(0xCD9E8D57u, c2, hi1, lo1);
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

GGP_HD int ggp_popc32(uint32_t v) {
#if defined(__CUDA_ARCH__)
    return __popc(v);
#else
    return __builtin_popcount(v);
#endif
}

// two standard normals of counter (c0, c1, c2, purpose | attempt): the polar method on v = 2 u - 1, u = 53 bits / 2^53 (exact)
GGP_HD void ggp_sim_normal2(uint64_t seed, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t purpose, const GgpMathTables* __restrict__ T,
                            double& z0, double& z1) {
    for (uint32_t attempt = 0;; ++attempt) {   // a call is rejected with probability 1 - pi / 4
        const uint32_t ctr[4] = {c0, c1, c2, (purpose << 24) | (attempt & 0xffffffu)};
        uint32_t w[4];
        ggp_philox4x32_10(ctr, seed, w);
        const double v1 = (double)(((uint64_t)w[0] << 21) | (w[1] >> 11)) * 0x1p-52 - 1.0;
        const double v2 = (double)(((uint64_t)w[2] << 21) | (w[3] >> 11)) * 0x1p-52 - 1.0;
        const double s = v1 * v1 + v2 * v2;
        if (s < 1.0 && s > 0.0) {
            const double f = GGP_SQRT(-2.0 * ggp_log(s, T) / s);
            z0 = v1 * f;
            z1 = v2 * f;
            return;
        }
    }
}

// Binomial(n, 1/2) for n <= 2^32: the popcount of the first n bits of the blocks (c0, BEFORE_FIRST, b >> 24, BITS << 24 | b & 0xffffff)
GGP_HD double ggp_sim_binomial_half(uint64_t seed, uint32_t c0, uint64_t n) {
    uint64_t k = 0;
    for (uint64_t b = 0; b * 128 < n; ++b) {
        const uint32_t ctr[4] = {c0, GGP_SIM_BEFORE_FIRST, (uint32_t)(b >> 24), ((uint32_t)GGP_SIM_BITS << 24) | (uint32_t)(b & 0xffffffu)};
        uint32_t w[4];
        ggp_philox4x32_10(ctr, seed, w);
        const uint64_t left = n - b * 128;
        for (int i = 0; i < 4; ++i) {
            const uint64_t take = left > (uint64_t)(32 * i) ? left - 32 * i : 0;
            if (take == 0) break;
            k += (uint64_t)ggp_popc32(take >= 32 ? w[i] : (w[i] & ((1u << take) - 1u)));
        }
    }
    return (double)k;
}

// the state z = (x, g, lambda, q) over dt in `substeps` sub-intervals with parameters p; OU draws at (c0, c1, sub-interval)
GGP_HD void ggp_sim_integrate(double* z, double dt, const double* __restrict__ p, int substeps, uint64_t seed, uint32_t c0, uint32_t c1,
                              const GgpMathTables* __restrict__ T) {
    const double h = dt / substeps;
    const double el = ggp_exp(-p[1] * h, T), eq = ggp_exp(-p[4] * h, T);
    const double sdl = GGP_SQRT(p[2] / (2.0 * p[1]) * (1.0 - el * el));
    const double sdq = GGP_SQRT(p[5] / (2.0 * p[4]) * (1.0 - eq * eq));
    for (int k = 0; k < substeps; ++k) {
        z[1] = z[1] + (ggp_exp(z[0], T) * z[3] - p[6] * z[1]) * h;
        z[0] = z[0] + z[2] * h;
        double n0, n1;
        ggp_sim_normal2(seed, c0, c1, (uint32_t)k, GGP_SIM_OU, T, n0, n1);
        z[2] = p[0] + (z[2] - p[0]) * el + sdl * n0;
        z[3] = p[3] + (z[3] - p[3]) * eq + sdq * n1;
    }
}

// the first time of the daughters of `slot` (the earlier of two)
GGP_HD double ggp_sim_division_time(const GgpDevForest& F, int slot) {
    const int d1 = F.s_d1[slot], d2 = F.s_d2[slot];
    const double t1 = d1 >= 0 ? F.time[F.s_off[d1]] : F.time[F.s_off[d2]];
    const double t2 = d2 >= 0 ? F.time[F.s_off[d2]] : t1;
    return t2 < t1 ? t2 : t1;
}

// one cell: its observations into x_out / g_out and edge, and (a mother) her state at the division time into end
GGP_HD void ggp_sim_cell(const GgpDevForest& F, const GgpSimArgs& A, int slot, const GgpMathTables* __restrict__ T) {
    const int64_t off = F.s_off[slot], N = F.n_cells;
    const int n = F.s_n[slot];
    const int parent = F.s_parent[slot];
    const int32_t cell = F.s_cell[slot];
    const uint32_t c0 = (uint32_t)(A.key ? A.key[cell] : cell);
    double z[4], n0, n1;
    if (parent < 0) {
        const double* p = A.params + GGP_NP * F.seg[off];
        ggp_sim_normal2(A.seed, c0, 0, 0, GGP_SIM_ROOT_XG, T, n0, n1);
        z[0] = A.root[0] + GGP_SQRT(A.root[2]) * n0;
        z[1] = A.root[1] + GGP_SQRT(A.root[3]) * n1;
        ggp_sim_normal2(A.seed, c0, 0, 0, GGP_SIM_ROOT_LQ, T, n0, n1);
        z[2] = p[0] + GGP_SQRT(p[2] / (2.0 * p[1])) * n0;
        z[3] = p[3] + GGP_SQRT(p[5] / (2.0 * p[4])) * n1;
    } else {
        for (int k = 0; k < 4; ++k) z[k] = A.end[k * N + parent];
        const double* pm = A.params + GGP_NP * F.seg[F.s_off[parent] + F.s_n[parent] - 1];
        const double rest = F.time[off] - ggp_sim_division_time(F, parent);
        if (rest > 0.0) ggp_sim_integrate(z, rest, pm, A.substeps, A.seed, c0, GGP_SIM_BEFORE_FIRST, T);
        ggp_sim_normal2(A.seed, c0, GGP_SIM_BEFORE_FIRST, 0, GGP_SIM_DIV, T, n0, n1);
        z[0] = z[0] - 0.6931471805599453 + GGP_SQRT(pm[9]) * n0;
        if (F.model.division_binomial) {
            const double r = rint(z[1] / pm[10]);
            z[1] = r <= 4294967296.0 ? pm[10] * ggp_sim_binomial_half(A.seed, c0, r > 1.0 ? (uint64_t)r : 1) : (double)NAN;
        } else {
            z[1] = z[1] / 2.0 + GGP_SQRT(pm[10]) * n1;
        }
    }
    for (int t = 0; t < n; ++t) {
        const double* p = A.params + GGP_NP * F.seg[off + t];
        ggp_sim_normal2(A.seed, c0, (uint32_t)t, 0, GGP_SIM_OBS, T, n0, n1);
        const double xo = z[0] + GGP_SQRT(p[7]) * n0;
        const double ga = z[1] + F.model.fp_auto;
        const double go = z[1] + GGP_SQRT(F.model.noise_scaled ? p[8] * (ga > 0.0 ? ga : 0.0) : p[8]) * n1;
        A.x_out[off + t] = xo;
        A.g_out[off + t] = go;
        if (!(xo - xo == 0.0 && go - go == 0.0)) {
#if defined(__CUDA_ARCH__)
            atomicMin(A.bad_key, (unsigned long long)c0);
#else
            if ((unsigned long long)c0 < *A.bad_key) *A.bad_key = c0;
#endif
        }
        if (t == 0) { A.edge[cell] = xo; A.edge[2 * N + cell] = go; }
        if (t == n - 1) { A.edge[N + cell] = xo; A.edge[3 * N + cell] = go; }
        if (t + 1 < n) ggp_sim_integrate(z, F.time[off + t + 1] - F.time[off + t], p, A.substeps, A.seed, c0, (uint32_t)t, T);
        else if (F.s_d1[slot] >= 0 || F.s_d2[slot] >= 0) {
            ggp_sim_integrate(z, ggp_sim_division_time(F, slot) - F.time[off + t], p, A.substeps, A.seed, c0, (uint32_t)t, T);
            for (int k = 0; k < 4; ++k) A.end[k * N + slot] = z[k];
        }
    }
}

#if defined(__CUDACC__)
#include "ggp_kernels.cuh"

// cells [slot0, slot0 + n_slots) of one generation, one thread each; the math tables staged in dynamic shared memory
__global__ void __launch_bounds__(GGP_SIM_BLOCK) ggp_sim_kernel(const GgpDevForest F, const GgpSimArgs A) {
    GgpMathTables& T = *reinterpret_cast<GgpMathTables*>(ggp_smem);
    ggp_stage_tables(&T);
    const int i = (int)(blockIdx.x * GGP_SIM_BLOCK + threadIdx.x);
    if (i < A.n_slots) ggp_sim_cell(F, A, A.slot0 + i, &T);
}
#endif
