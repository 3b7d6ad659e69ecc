// tests/hostcheck/gradcheck.cpp — the gradient of the FAST log-likelihood on the host: the dual-number evaluation of
// ggp_fast.cuh (gfp_gaussian_process_b200/csrc/ggp_dual.cuh) in double, which is the device gradient kernel's arithmetic up to
// FMA contraction, and the binary128 central difference of the 16-node binary128 evaluation, the truth it is measured against.
// Test infrastructure (tests/test_grad_host.py, tests/test_gpu_grad.py, tools/grad_check.py); not part of the product.
#include "fastcheck.cpp"

#include "../../gfp_gaussian_process_b200/csrc/ggp_dual.cuh"

// total log-likelihood of the forest for one parameter vector (any scalar type); clears `valid` like ggp_fast_cell
template <class T, int N, class GL>
static T forest_total(const GgpLayout& L, const GgpDevForest& F, const T* p, const GL& gln, bool& valid) {
    std::vector<GgpFastState<T>> state((size_t)L.n_cells);
    GgpFastConstsOnDemand<T, N, GL> kp(F, p, gln);
    T total = T(0);
    for (int64_t slot = 0; slot < L.n_cells; ++slot) {
        GgpFastState<T> s;
        if (F.s_parent[slot] >= 0) s = state[(size_t)F.s_parent[slot]];
        total += ggp_fast_cell<T, N>(F, (int)slot, p, s, kp, valid);
        state[(size_t)slot] = s;
    }
    return total;
}

template <int N>
static int run_dual(const ggp_forest_desc* d, const double* params, int n_vec, double* out_total, double* out_grad, int* out_valid) {
    typedef GgpDual<GGP_NP> T;
    GgpLayout L;
    if (!L.build(d).empty()) return -1;
    const GgpDevForest F = fc_dev(L, d);
    for (int v = 0; v < n_vec; ++v) {
        T p[GGP_NP];
        for (int i = 0; i < GGP_NP; ++i) {
            p[i] = T(params[GGP_NP * v + i]);
            p[i].d[i] = 1.0;
        }
        bool valid = true;
        const T total = forest_total<T, N>(L, F, p, DoubleGL<N>(), valid);
        out_total[v] = total.v;
        for (int i = 0; i < GGP_NP; ++i) out_grad[(size_t)GGP_NP * v + i] = total.d[i];
        out_valid[v] = valid ? 1 : 0;
    }
    return 0;
}

extern "C" {
// value and all 11 derivatives of the fast log-likelihood (dual numbers in double), n_nodes in {3,4,5,6,8,10,12,16};
// out_total [n_vec], out_grad [n_vec][11], out_valid [n_vec]
int gc_loglik_grad(const ggp_forest_desc* d, const double* params, int n_vec, int n_nodes, double* out_total, double* out_grad,
                   int* out_valid) {
    switch (n_nodes) {
        case 3: return run_dual<3>(d, params, n_vec, out_total, out_grad, out_valid);
        case 4: return run_dual<4>(d, params, n_vec, out_total, out_grad, out_valid);
        case 5: return run_dual<5>(d, params, n_vec, out_total, out_grad, out_valid);
        case 6: return run_dual<6>(d, params, n_vec, out_total, out_grad, out_valid);
        case 8: return run_dual<8>(d, params, n_vec, out_total, out_grad, out_valid);
        case 10: return run_dual<10>(d, params, n_vec, out_total, out_grad, out_valid);
        case 12: return run_dual<12>(d, params, n_vec, out_total, out_grad, out_valid);
        case 16: return run_dual<16>(d, params, n_vec, out_total, out_grad, out_valid);
    }
    return -2;
}

// central difference of the binary128 16-node evaluation along every parameter with step h_i = rel_step |p_i|, the difference
// taken in binary128 and only the quotient rounded to double; out_total [n_vec] the binary128 value, out_grad [n_vec][11]
int gc_grad_quad(const ggp_forest_desc* d, const double* params, int n_vec, double rel_step, double* out_total, double* out_grad,
                 int* out_valid) {
    GgpLayout L;
    if (!L.build(d).empty()) return -1;
    const GgpDevForest F = fc_dev(L, d);
    const QuadGL gln(16);
    for (int v = 0; v < n_vec; ++v) {
        quad p[GGP_NP];
        for (int i = 0; i < GGP_NP; ++i) p[i] = (quad)params[GGP_NP * v + i];
        bool valid = true;
        out_total[v] = (double)forest_total<quad, 16>(L, F, p, gln, valid);
        for (int i = 0; i < GGP_NP; ++i) {
            const quad x = p[i], h = (quad)rel_step * fabsq(x);
            p[i] = x + h;
            const quad up = forest_total<quad, 16>(L, F, p, gln, valid);
            p[i] = x - h;
            const quad dn = forest_total<quad, 16>(L, F, p, gln, valid);
            p[i] = x;
            out_grad[(size_t)GGP_NP * v + i] = (double)((up - dn) / (2 * h));
        }
        out_valid[v] = valid ? 1 : 0;
    }
    return 0;
}
}
