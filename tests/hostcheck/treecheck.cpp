// tests/hostcheck/treecheck.cpp — per-tree scores of the FAST log-likelihood on the host: the dual-number evaluation of
// gradcheck.cpp with every cell's value and derivatives added into its lineage tree (trees numbered as the library numbers
// them: roots in cell order), and the binary128 central difference of every tree's 16-node binary128 log-likelihood, the truth.
// Test infrastructure (tests/test_tree_host.py, tests/test_gpu_tree.py); not part of the product.
#include "gradcheck.cpp"

// tree of every slot (slots in generation order: a mother's slot comes before her daughters')
static std::vector<int32_t> tree_of_slot(const GgpLayout& L) {
    std::vector<int32_t> t((size_t)L.n_cells);
    for (int64_t s = 0; s < L.n_cells; ++s) t[(size_t)s] = L.s_parent[s] < 0 ? L.s_root[s] : t[(size_t)L.s_parent[s]];
    return t;
}

static double value_of(const GgpDual<GGP_NP>& x) { return x.v; }
static double value_of(quad x) { return (double)x; }

// every tree's log-likelihood out[n_roots] (any scalar type) and, if abs_out, the sum of |cell log-likelihood| over its cells
template <class T, int N, class GL>
static void forest_trees(const GgpLayout& L, const GgpDevForest& F, const T* p, const GL& gln, T* out, double* abs_out, bool& valid) {
    const std::vector<int32_t> tree = tree_of_slot(L);
    std::vector<GgpFastState<T>> state((size_t)L.n_cells);
    GgpFastConstsOnDemand<T, N, GL> kp(F, p, gln);
    for (int32_t t = 0; t < L.n_roots; ++t) {
        out[t] = T(0);
        if (abs_out) abs_out[t] = 0.0;
    }
    for (int64_t slot = 0; slot < L.n_cells; ++slot) {
        GgpFastState<T> s;
        if (F.s_parent[slot] >= 0) s = state[(size_t)F.s_parent[slot]];
        const T own = ggp_fast_cell<T, N>(F, (int)slot, p, s, kp, valid);
        out[tree[(size_t)slot]] += own;
        if (abs_out) abs_out[tree[(size_t)slot]] += std::fabs(value_of(own));
        state[(size_t)slot] = s;
    }
}

template <int N>
static int run_trees(const ggp_forest_desc* d, const double* params, int n_vec, double* out_ll, double* out_grad, double* out_abs,
                     int* out_valid) {
    typedef GgpDual<GGP_NP> T;
    GgpLayout L;
    if (!L.build(d).empty()) return -1;
    const GgpDevForest F = fc_dev(L, d);
    const size_t R = (size_t)L.n_roots;
    std::vector<T> tr(R);
    for (int v = 0; v < n_vec; ++v) {
        T p[GGP_NP];
        for (int i = 0; i < GGP_NP; ++i) {
            p[i] = T(params[GGP_NP * v + i]);
            p[i].d[i] = 1.0;
        }
        bool valid = true;
        forest_trees<T, N>(L, F, p, DoubleGL<N>(), tr.data(), out_abs + v * R, valid);
        for (size_t t = 0; t < R; ++t) {
            out_ll[v * R + t] = tr[t].v;
            for (int i = 0; i < GGP_NP; ++i) out_grad[(v * R + t) * GGP_NP + i] = tr[t].d[i];
        }
        out_valid[v] = valid ? 1 : 0;
    }
    return 0;
}

extern "C" {
// every tree's value and 11 derivatives of the fast log-likelihood (dual numbers in double), n_nodes in {4,5,6,8,10};
// out_ll [n_vec][n_roots], out_grad [n_vec][n_roots][11], out_abs [n_vec][n_roots] sum of |cell log-likelihood|, out_valid [n_vec]
int tc_tree_grad(const ggp_forest_desc* d, const double* params, int n_vec, int n_nodes, double* out_ll, double* out_grad,
                 double* out_abs, int* out_valid) {
    switch (n_nodes) {
        case 4: return run_trees<4>(d, params, n_vec, out_ll, out_grad, out_abs, out_valid);
        case 5: return run_trees<5>(d, params, n_vec, out_ll, out_grad, out_abs, out_valid);
        case 6: return run_trees<6>(d, params, n_vec, out_ll, out_grad, out_abs, out_valid);
        case 8: return run_trees<8>(d, params, n_vec, out_ll, out_grad, out_abs, out_valid);
        case 10: return run_trees<10>(d, params, n_vec, out_ll, out_grad, out_abs, out_valid);
    }
    return -2;
}

// every tree's binary128 16-node log-likelihood and its central differences along every parameter with step h_i = rel_step |p_i|,
// differenced in binary128; out_ll [n_vec][n_roots], out_grad [n_vec][n_roots][11]
int tc_tree_quad(const ggp_forest_desc* d, const double* params, int n_vec, double rel_step, double* out_ll, double* out_grad,
                 int* out_valid) {
    GgpLayout L;
    if (!L.build(d).empty()) return -1;
    const GgpDevForest F = fc_dev(L, d);
    const QuadGL gln(16);
    const size_t R = (size_t)L.n_roots;
    std::vector<quad> tr(R), up(R), dn(R);
    for (int v = 0; v < n_vec; ++v) {
        quad p[GGP_NP];
        for (int i = 0; i < GGP_NP; ++i) p[i] = (quad)params[GGP_NP * v + i];
        bool valid = true;
        forest_trees<quad, 16>(L, F, p, gln, tr.data(), nullptr, valid);
        for (size_t t = 0; t < R; ++t) out_ll[v * R + t] = (double)tr[t];
        for (int i = 0; i < GGP_NP; ++i) {
            const quad x = p[i], h = (quad)rel_step * fabsq(x);
            p[i] = x + h;
            forest_trees<quad, 16>(L, F, p, gln, up.data(), nullptr, valid);
            p[i] = x - h;
            forest_trees<quad, 16>(L, F, p, gln, dn.data(), nullptr, valid);
            p[i] = x;
            for (size_t t = 0; t < R; ++t) out_grad[(v * R + t) * GGP_NP + i] = (double)((up[t] - dn[t]) / (2 * h));
        }
        out_valid[v] = valid ? 1 : 0;
    }
    return 0;
}
}
