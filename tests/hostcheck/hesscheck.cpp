// tests/hostcheck/hesscheck.cpp — the Hessian of the FAST log-likelihood on the host: the second-order Taylor evaluation
// (GgpTaylor2, gfp_gaussian_process_b200/csrc/ggp_dual.cuh) of ggp_fast.cuh in double through the library's own evaluation plan
// (GgpEvalPlan, ggp_types.cuh: the evaluations, their seeding and the unscaling), which is the device Hessian kernels'
// arithmetic up to FMA contraction, and binary128 second differences of the 16-node binary128 evaluation, the truth it is
// measured against (they share no code with the Taylor numbers).
// Test infrastructure (tests/test_hess_host.py, tests/test_gpu_hess.py, tools/grad_check.py); not part of the product.
#include "gradcheck.cpp"   // forest_total, the binary128 rule and the dual-number helpers

// value, gradient [n_dirs] and Hessian [n_dirs][n_dirs] of the fast log-likelihood over the directions dirs with GgpTaylor2 in
// double: every evaluation of the order-2 plan, seeded as the device seeds it, then the plan's unscaling; out_valid [n_vec]:
// every evaluation stayed inside the rule's validity range
template <int N>
static int run_taylor2(const ggp_forest_desc* d, const double* params, int n_vec, const int* dirs, int n, double* out_total,
                       double* out_grad, double* out_hess, int* out_valid) {
    typedef GgpTaylor2 T;
    GgpLayout L;
    if (!L.build(d).empty()) return -1;
    const GgpDevForest F = fc_dev(L, d);
    GgpEvalPlan P{};
    P.order = 2;
    P.n_dirs = n;
    for (int k = 0; k < n; ++k) P.dirs[k] = dirs[k];
    P.select(0, P.evals());
    std::vector<double> o((size_t)P.evals() * P.comps());
    for (int v = 0; v < n_vec; ++v) {
        const double* pv = params + (size_t)GGP_NP * v;
        bool valid = true;
        for (int e = 0; e < P.evals(); ++e) {
            T p[GGP_NP];
            for (int i = 0; i < GGP_NP; ++i) p[i] = T(pv[i], P.seeds(e, i) ? ggp_hess_scale(pv[i]) : 0.0, 0.0);
            T total = forest_total<T, N>(L, F, p, DoubleGL<N>(), valid);
            for (int j = 0; j < P.comps(); ++j) o[(size_t)e * P.comps() + j] = ggp_comp(total, j);
        }
        out_total[v] = o[0];
        P.unscale(pv, o.data(), out_grad + (size_t)n * v, out_hess + (size_t)n * n * v);
        out_valid[v] = valid ? 1 : 0;
    }
    return 0;
}

extern "C" {
// second differences of the binary128 16-node evaluation over the directions dirs with steps h_i = rel_step |p_i|, differenced
// in binary128 and only the quotient rounded to double: H_ii = (f(+h_i) - 2 f + f(-h_i)) / h_i^2, H_ij = (f(++) - f(+-) - f(-+)
// + f(--)) / (4 h_i h_j); 1 + 2 n + 2 n (n - 1) evaluations.  out_total [n_vec] the binary128 value, out_hess [n_vec][n][n]
int gc_hess_quad(const ggp_forest_desc* d, const double* params, int n_vec, double rel_step, const int* dirs, int n, double* out_total,
                 double* out_hess, int* out_valid) {
    GgpLayout L;
    if (!L.build(d).empty()) return -1;
    const GgpDevForest F = fc_dev(L, d);
    const QuadGL gln(16);
    for (int v = 0; v < n_vec; ++v) {
        quad p[GGP_NP];
        for (int i = 0; i < GGP_NP; ++i) p[i] = (quad)params[GGP_NP * v + i];
        bool valid = true;
        const quad f0 = forest_total<quad, 16>(L, F, p, gln, valid);
        out_total[v] = (double)f0;
        double* H = out_hess + (size_t)n * n * v;
        for (int a = 0; a < n; ++a) {
            const int i = dirs[a];
            const quad xi = p[i], hi = (quad)rel_step * fabsq(xi);
            p[i] = xi + hi;
            const quad up = forest_total<quad, 16>(L, F, p, gln, valid);
            p[i] = xi - hi;
            const quad dn = forest_total<quad, 16>(L, F, p, gln, valid);
            p[i] = xi;
            H[(size_t)a * n + a] = (double)((up - 2 * f0 + dn) / (hi * hi));
            for (int b = a + 1; b < n; ++b) {
                const int j = dirs[b];
                const quad xj = p[j], hj = (quad)rel_step * fabsq(xj);
                quad f[4];
                for (int c = 0; c < 4; ++c) {
                    p[i] = (c & 2) ? xi - hi : xi + hi;
                    p[j] = (c & 1) ? xj - hj : xj + hj;
                    f[c] = forest_total<quad, 16>(L, F, p, gln, valid);
                }
                p[i] = xi;
                p[j] = xj;
                H[(size_t)a * n + b] = H[(size_t)b * n + a] = (double)((f[0] - f[1] - f[2] + f[3]) / (4 * hi * hj));
            }
        }
        out_valid[v] = valid ? 1 : 0;
    }
    return 0;
}

// value, gradient and Hessian of the GgpTaylor2 evaluation in double (run_taylor2), n_nodes in {3,4,5,6,8,10,12,16}
int gc_loglik_hess(const ggp_forest_desc* d, const double* params, int n_vec, int n_nodes, const int* dirs, int n_dirs, double* out_total,
                   double* out_grad, double* out_hess, int* out_valid) {
    switch (n_nodes) {
        case 3: return run_taylor2<3>(d, params, n_vec, dirs, n_dirs, out_total, out_grad, out_hess, out_valid);
        case 4: return run_taylor2<4>(d, params, n_vec, dirs, n_dirs, out_total, out_grad, out_hess, out_valid);
        case 5: return run_taylor2<5>(d, params, n_vec, dirs, n_dirs, out_total, out_grad, out_hess, out_valid);
        case 6: return run_taylor2<6>(d, params, n_vec, dirs, n_dirs, out_total, out_grad, out_hess, out_valid);
        case 8: return run_taylor2<8>(d, params, n_vec, dirs, n_dirs, out_total, out_grad, out_hess, out_valid);
        case 10: return run_taylor2<10>(d, params, n_vec, dirs, n_dirs, out_total, out_grad, out_hess, out_valid);
        case 12: return run_taylor2<12>(d, params, n_vec, dirs, n_dirs, out_total, out_grad, out_hess, out_valid);
        case 16: return run_taylor2<16>(d, params, n_vec, dirs, n_dirs, out_total, out_grad, out_hess, out_valid);
    }
    return -2;
}
}
