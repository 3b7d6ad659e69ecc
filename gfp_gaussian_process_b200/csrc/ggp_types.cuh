// ggp_types.cuh — host/device function qualifiers and the plain structs shared by every translation unit of the library:
// the strict kernels (ggp_b200.cu, compiled with -fmad=false) and the fast likelihood kernels (ggp_fast.cu, -fmad=true).
// No kernels, no device variables: safe to include from several translation units.
#pragma once
#include <stdint.h>
#include <math.h>

#if defined(__CUDACC__)
#define GGP_HD __host__ __device__ __forceinline__
#define GGP_HD_NOINLINE static __host__ __device__ __noinline__
#define GGP_HDM __host__ __device__ __forceinline__
#else
#define GGP_HD static inline
#define GGP_HD_NOINLINE static
#define GGP_HDM inline
#endif

struct GgpModel {          // what MOMAdata carries besides data (moma_input.h:44-47)
    int noise_scaled;      // noise_model == "scaled"
    int division_binomial; // cell_division_model == "binomial"
    double fp_auto;
};

#define GGP_NP 11
#define GGP_INLINE_VECS 8

struct GgpDevForest {
    int64_t n_cells, n_ctp;
    // measurements, caller's ctp order
    const double* time;
    const double* x;
    const double* g;
    const int32_t* seg;
    // per slot (generation order)
    const int64_t* s_off;     // first ctp
    const int32_t* s_n;       // number of points
    const int32_t* s_parent;  // parent slot or -1
    const int32_t* s_d1;      // daughter slots or -1
    const int32_t* s_d2;
    const int32_t* s_root;    // root number (cell order) or -1
    const int32_t* s_cell;    // caller's cell index
    const int64_t* s_dfs0;    // rank of the cell's first ctp in the reference's depth-first order
    GgpModel model;
    double init_f[4], init_r[4];
    // fast likelihood only: index into the forest's table of distinct time steps, per time point = the step that arrives
    // there (from the previous point of the cell, or from the mother's last point); 0xffff at a root's first point
    const uint16_t* dt_idx;
    int32_t n_dt;
};

struct GgpFwdArgs {
    int slot0, n_slots;          // this generation
    const double* params;        // LIK: [n_vec][11]; PRED: [n_seg][11]
    int v0, v_count;             // vectors of this chunk
    double* carry;               // CHAIN: [n_roots][16] in/out
    double* state;               // SoA [14][v_count * n_cells] end-of-cell posteriors (upper triangle)
    double* partial;             // [v_count][n_partial]
    int partial0, n_partial;     // first partial of this launch, partials per vector
    double* cell_ll;             // NULL or [n_vec][n_cells] (caller's cell order)
    unsigned long long* nan_key; // [n_vec] min depth-first ctp rank with a NaN term
    double* out_fwd;             // PRED: [n_ctp][20]
    int n_seg;                   // PRED: number of parameter sets
    // LIK, params == nullptr: up to GGP_INLINE_VECS parameter vectors travel in the launch arguments (an evaluation that
    // runs behind a streamed upload must not queue a copy, or read host memory, behind the upload's DMA traffic)
    double inline_params[GGP_INLINE_VECS * GGP_NP];
};

struct GgpBwdArgs {
    int slot0, n_slots;
    const double* params;   // [n_seg][11]
    const double* fwd;      // [n_ctp][20] forward posteriors (a leaf starts from the stale one at its last point)
    double* bwd;            // [n_ctp][20] out
    double* bstate;         // [n_cells][20] by slot: MOMAdata::mean/cov after the backward pass (sign-flipped frame)
    int n_seg;              // number of parameter sets
};

// the scale s of a parameter p along which the Hessian's evaluations step (DESIGN.md 5.7): the power of two nearest |p|, 1 for
// p = 0 (or a non-finite p).  A power of two keeps the scaling and the unscaling exact; the device seeds with it and the host
// divides by it, so both take it from here
GGP_HDM double ggp_hess_scale(double p) {
    const double a = fabs(p);
    if (!(a > 0.0) || a - a != 0.0) return 1.0;
    int e;
    const double m = frexp(a, &e);   // a = m 2^e, 0.5 <= m < 1: the nearer of 2^(e-1) and 2^e
    return ldexp(1.0, m >= 0.75 ? e : e - 1);
}

// the evaluations of one parameter vector on the fast path (DESIGN.md 5.4, 5.6, 5.7), along the directions dirs (distinct
// parameter indices):
//   order 0: the log-likelihood; one evaluation, result (value);
//   order 1: the gradient; one evaluation per direction k, seeding e_k; results (value, g_k);
//   order 2: value, gradient and Hessian by polarization; one evaluation per pair k <= l of directions (k-major: (0,0), (0,1) ..
//            (0,n-1), (1,1) ..), stepping along s_k e_k + s_l e_l (s_k e_k once if k == l) with the scales s = ggp_hess_scale of
//            the vector's parameters; results (value, g.u, u^T H u).
// A launch runs the evaluations select() picked: its evaluation e seeds the parameters a[e] and b[e] (one if a[e] == b[e]).
#define GGP_MAX_EVALS (GGP_NP * (GGP_NP + 1) / 2)
struct GgpEvalPlan {
    int32_t order;
    int32_t n_dirs;
    int32_t dirs[GGP_NP];
    int32_t n_run;
    int8_t a[GGP_MAX_EVALS], b[GGP_MAX_EVALS];

    // evaluations per vector and results per evaluation
    GGP_HDM int evals() const { return order == 0 ? 1 : order == 1 ? n_dirs : n_dirs * (n_dirs + 1) / 2; }
    GGP_HDM int comps() const { return order + 1; }
    // the evaluation of directions k <= l
    GGP_HDM int pair(int k, int l) const { return order == 1 ? k : k * n_dirs - k * (k - 1) / 2 + (l - k); }
    GGP_HDM bool seeds(int e, int i) const { return a[e] == i || b[e] == i; }
    // the launch runs evaluations [e0, e0 + ec)
    void select(int e0, int ec) {
        n_run = ec;
        for (int k = 0; k < n_dirs; ++k)
            for (int l = k; l < (order == 2 ? n_dirs : k + 1); ++l) {
                const int e = pair(k, l) - e0;
                if (e >= 0 && e < ec) { a[e] = (int8_t)dirs[k]; b[e] = (int8_t)dirs[l]; }
            }
    }
    // the gradient row [n_dirs] and (order 2) the Hessian block [n_dirs][n_dirs] of one vector from the results o [evals][comps]
    // of its evaluations; p: its parameters.  Order 2 undoes the polarization: with dd_kl = u^T H u of evaluation (k, l),
    // g_k = d_kk / s_k, H_kk = dd_kk / s_k^2, H_kl = H_lk = (dd_kl - dd_kk - dd_ll) / (2 s_k s_l); every division is by a power of two
    void unscale(const double* p, const double* o, double* grad, double* hess) const {
        const int n = n_dirs, C = comps();
        for (int k = 0; k < n; ++k) {
            const double sk = order == 2 ? ggp_hess_scale(p[dirs[k]]) : 1.0;
            const double* ok = o + pair(k, k) * C;
            grad[k] = ok[1] / sk;
            if (order == 1) continue;
            hess[k * n + k] = ok[2] / (sk * sk);
            for (int l = k + 1; l < n; ++l) {
                const double sl = ggp_hess_scale(p[dirs[l]]);
                const double ol = o[pair(l, l) * C + 2];
                // the diagonal term of the smaller parameter index first: the same bits whatever the order of dirs
                const bool kf = dirs[k] < dirs[l];
                const double h = (o[pair(k, l) * C + 2] - (kf ? ok[2] : ol) - (kf ? ol : ok[2])) / (2.0 * sk * sl);
                hess[k * n + l] = hess[l * n + k] = h;
            }
        }
    }
};
