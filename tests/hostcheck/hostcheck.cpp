// tests/hostcheck/hostcheck.cpp — compiles the product's host+device math headers FOR THE HOST
// (g++ -ffp-contract=off) so that CPU-only tests can compare them bit-for-bit against the
// reference build (oracle/_ref) and the host libm.  Test infrastructure; not part of the product.
#include "../../gfp_gaussian_process_b200/csrc/ggp_tables_data.h"
#include "../../gfp_gaussian_process_b200/csrc/ggp_dawson.cuh"
#include "../../gfp_gaussian_process_b200/csrc/ggp_step.cuh"
#include "../../gfp_gaussian_process_b200/csrc/ggp_filter.cuh"
#include "../../gfp_gaussian_process_b200/csrc/ggp_linalg.cuh"

static const GgpMathTables g_tables = GGP_MATH_TABLES_INIT;

extern "C" {
void hc_exp(long n, const double* x, double* y) { for (long i = 0; i < n; ++i) y[i] = ggp_exp(x[i], &g_tables); }
void hc_log(long n, const double* x, double* y) { for (long i = 0; i < n; ++i) y[i] = ggp_log(x[i], &g_tables); }
void hc_pow(long n, const double* x, const double* e, double* y) { for (long i = 0; i < n; ++i) y[i] = ggp_pow(x[i], e[i], &g_tables); }
// the log-evidence term from the quadratic form on (ggp_filter.cuh::ggp_log_evidence_finish): in5 [n][5] = qf, S00, S01, S10, S11
void hc_ll_finish(long n, const double* in5, double* y) {
    for (long i = 0; i < n; ++i) y[i] = ggp_log_evidence_finish(in5[5 * i], in5[5 * i + 1], in5[5 * i + 2], in5[5 * i + 3], in5[5 * i + 4], &g_tables);
}
void hc_dawson(long n, const double* x, double* y) { for (long i = 0; i < n; ++i) y[i] = ggp_dawson(x[i], &g_tables); }
// state = 4 means + 10 upper-triangular covariances (xx,xg,xl,xq,gg,gl,gq,ll,lq,qq)
void hc_propagate(long n, const double* state14, const double* dt, const double* p7, double* out14) {
    for (long i = 0; i < n; ++i) {
        GgpState s;
        for (int k = 0; k < 4; ++k) s.m[k] = state14[14 * i + k];
        for (int k = 0; k < 10; ++k) s.c[k] = state14[14 * i + 4 + k];
        GgpOuParams p = {p7[0], p7[1], p7[2], p7[3], p7[4], p7[5], p7[6]};
        double scratch[GGP_SCRATCH];
        GgpScratch S{scratch, 1};
        ggp_propagate(s, dt[i], p, &g_tables, S);
        for (int k = 0; k < 4; ++k) out14[14 * i + k] = s.m[k];
        for (int k = 0; k < 10; ++k) out14[14 * i + 4 + k] = s.c[k];
    }
}
}

// ------------------------------------------------------------------------------------------------
// whole passes on the host: the product's per-cell bodies (ggp_cell.cuh) and layout (ggp_layout.hpp)
// driven in the same generation order as the kernels' launch sequence in ggp_b200.cu.
// ------------------------------------------------------------------------------------------------
#include "../../gfp_gaussian_process_b200/csrc/ggp_layout.hpp"
#include "../../gfp_gaussian_process_b200/csrc/ggp_cell.cuh"
#include "../../gfp_gaussian_process_b200/csrc/ggp_joints.cuh"
#include "../../gfp_gaussian_process_b200/csrc/ggp_coop.cuh"

static GgpDevForest hc_dev(const GgpLayout& L, const ggp_forest_desc* d) {
    GgpDevForest F;
    F.n_cells = L.n_cells; F.n_ctp = L.n_ctp;
    F.time = d->time; F.x = d->log_length; F.g = d->fp; F.seg = L.seg.data();
    F.s_off = L.s_off.data(); F.s_n = L.s_n.data(); F.s_parent = L.s_parent.data(); F.s_d1 = L.s_d1.data();
    F.s_d2 = L.s_d2.data(); F.s_root = L.s_root.data(); F.s_cell = L.s_cell.data(); F.s_dfs0 = L.s_dfs0.data();
    F.model.noise_scaled = d->noise_model == GGP_NOISE_SCALED;
    F.model.division_binomial = d->division_model == GGP_DIVISION_BINOMIAL;
    F.model.fp_auto = d->fp_auto;
    for (int i = 0; i < 4; ++i) { F.init_f[i] = L.init_f[i]; F.init_r[i] = L.init_r[i]; }
    return F;
}

extern "C" {

// returns 0 or -1 (layout error); out_cell_ll [n_vec][n_cells]; carry NULL or [n_roots][16] in/out;
// nan_rank [n_vec] = depth-first ctp rank of the first NaN term or -1
int hc_loglik(const ggp_forest_desc* d, const double* params, int n_vec, double* carry, double* out_cell_ll, long long* nan_rank) {
    GgpLayout L;
    if (!L.build(d).empty()) return -1;
    double scratch[GGP_SCRATCH];
    const GgpScratch S{scratch, 1};
    const GgpDevForest F = hc_dev(L, d);
    std::vector<double> state((size_t)14 * n_vec * L.n_cells);
    std::vector<unsigned long long> nan(n_vec, ~0ull);
    GgpFwdArgs A{};
    A.params = params; A.v0 = 0; A.v_count = n_vec; A.carry = carry; A.state = state.data();
    A.cell_ll = out_cell_ll; A.nan_key = nan.data();
    for (int g = 0; g < L.n_gen; ++g)
        for (int64_t s = L.gen_start[g]; s < L.gen_start[g + 1]; ++s) {
            if (g == 0 && carry) {
                double Cc[16];
                for (int i = 0; i < 16; ++i) Cc[i] = carry[16 * L.s_root[s] + i];
                for (int v = 0; v < n_vec; ++v) ggp_cell_forward<false, true>(F, A, (int)s, v, params + 11 * v, &g_tables, S, Cc);
                for (int i = 0; i < 16; ++i) carry[16 * L.s_root[s] + i] = Cc[i];
            } else {
                for (int v = 0; v < n_vec; ++v) ggp_cell_forward<false, false>(F, A, (int)s, v, params + 11 * v, &g_tables, S, nullptr);
            }
        }
    for (int v = 0; v < n_vec; ++v) nan_rank[v] = nan[v] == ~0ull ? -1 : (long long)nan[v];
    return 0;
}

// upload chunks of the layout (ggp_layout.hpp): ctp_chunk_start [n_chunks+1], chunk of every cell [n_cells] (from the
// per-generation slot ranges), returns the number of chunks or -1
int hc_layout_chunks(const ggp_forest_desc* d, int want_chunks, const double* fractions, long long* ctp_chunk_start, int* chunk_of_cell) {
    GgpLayout L;
    if (!L.build(d, want_chunks, fractions).empty()) return -1;
    for (int k = 0; k <= L.n_chunks; ++k) ctp_chunk_start[k] = L.ctp_chunk_start[k];
    for (int g = 0; g < L.n_gen; ++g)
        for (int k = 0; k < L.n_chunks; ++k) {
            const int64_t* row = L.gen_chunk_start.data() + (size_t)g * (L.n_chunks + 1);
            for (int64_t s = row[k]; s < row[k + 1]; ++s) chunk_of_cell[L.cell_of_slot[s]] = k;
        }
    return L.n_chunks;
}
// the likelihood with the cooperative step (ggp_coop.cuh): the four roles of every phase run in sequence over one
// cell's scratch column, in the order of ggp_loglik_coop_kernel (ggp_coop_kernels.cuh).  fresh mode only.
int hc_loglik_coop(const ggp_forest_desc* d, const double* params, int n_vec, double* out_cell_ll, long long* nan_rank) {
    GgpLayout L;
    if (!L.build(d).empty()) return -1;
    double scratch[GGP_CS_COUNT];
    const GgpScratch S{scratch, 1};
    const GgpDevForest F = hc_dev(L, d);
    std::vector<double> state((size_t)14 * L.n_cells);
    for (int v = 0; v < n_vec; ++v) {
        const double* p = params + 11 * v;
        unsigned long long nan = ~0ull;
        for (int64_t slot = 0; slot < L.n_cells; ++slot) {
            const int64_t off = F.s_off[slot];
            const int n = F.s_n[slot], parent = F.s_parent[slot];
            double own = 0.0;
            int t = 0;
            int64_t from = off;
            if (parent < 0) {
                double mu[4], C[16];
                ggp_root_start(mu, C, nullptr, F, p, off, &g_tables, [&](double ll) {
                    own = own + ll;
                    if (ll != ll) GGP_NAN_MIN(&nan, F.s_dfs0[slot]);
                });
                GgpState s;
                ggp_state_from16(s, mu, C);
                for (int k = 0; k < 4; ++k) S[GGP_CS_ST + k] = s.m[k];
                for (int k = 0; k < 10; ++k) S[GGP_CS_ST + 4 + k] = s.c[k];
            } else {
                for (int k = 0; k < 14; ++k) S[GGP_CS_ST + k] = state[k * L.n_cells + parent];
                t = -1;
                from = F.s_off[parent] + F.s_n[parent] - 1;
            }
            bool pend = false;   // as in the kernel: phase 3 leaves the log-evidence term pending, the next phase 0 (or the tail) finishes it
            auto finish_pending = [&]() {
                const double ll = ggp_coop_ll_deferred(GGP_SLOTS_REF(S), &g_tables);
                own = own + ll;
                if (ll != ll) GGP_NAN_MIN(&nan, F.s_dfs0[slot] + t);
                pend = false;
            };
            while (t + 1 < n) {
                const double dt = F.time[off + t + 1] - F.time[from];
                for (int ph = 0; ph < GGP_COOP_PHASES; ++ph)
                    for (int role = 0; role < GGP_COOP_ROLES; ++role) {
                        if (ph == 0 && role == 0 && pend) {   // as in the kernel: the pending term is finished inside role 0's phase 0
                            double ll = 0.0;
                            ggp_coop_run_phase(0, 0, S, ggp_ou(p, false), dt, &g_tables, false, GGP_NO_GL3, &ll);
                            own = own + ll;
                            if (ll != ll) GGP_NAN_MIN(&nan, F.s_dfs0[slot] + t);
                            pend = false;
                        } else {
                            ggp_coop_run_phase(ph, role, S, ggp_ou(p, false), dt, &g_tables);
                        }
                    }
                const int64_t at = off + t + 1;
                for (int role = 0; role < GGP_COOP_ROLES; ++role) ggp_coop_ph3<true>(role, S, t < 0, p, F.x[at], F.g[at], F.model, &g_tables);
                ++t;
                from = at;
                pend = true;
            }
            if (pend) finish_pending();
            for (int k = 0; k < 14; ++k) state[k * L.n_cells + slot] = S[GGP_CS_ST + k];
            out_cell_ll[(int64_t)v * L.n_cells + F.s_cell[slot]] = own;
        }
        nan_rank[v] = nan == ~0ull ? -1 : (long long)nan;
    }
    return 0;
}

// fwd/bwd/comb [n_ctp][20]; bstate [n_cells][20] in the caller's cell order
int hc_predict(const ggp_forest_desc* d, const double* params, int n_seg, double* fwd, double* bwd, double* comb, double* bstate_cells) {
    GgpLayout L;
    if (!L.build(d).empty() || L.max_seg >= n_seg) return -1;
    double scratch[GGP_SCRATCH];
    const GgpScratch S{scratch, 1};
    const GgpDevForest F = hc_dev(L, d);
    std::vector<double> state((size_t)14 * L.n_cells), bstate((size_t)20 * L.n_cells);
    GgpFwdArgs A{};
    A.params = params; A.v_count = 1; A.state = state.data(); A.out_fwd = fwd;
    for (int64_t s = 0; s < L.n_cells; ++s) ggp_cell_forward<true, false>(F, A, (int)s, 0, nullptr, &g_tables, S, nullptr);
    GgpBwdArgs B{};
    B.params = params; B.fwd = fwd; B.bwd = bwd; B.bstate = bstate.data();
    for (int64_t s = L.n_cells - 1; s >= 0; --s) ggp_cell_backward(F, B, (int)s, &g_tables, S);
    for (int64_t i = 0; i < L.n_ctp; ++i) ggp_ctp_combine(fwd + 20 * i, bwd + 20 * i, params + 11 * L.comb_seg[i], comb + 20 * i);
    for (int64_t s = 0; s < L.n_cells; ++s)
        for (int k = 0; k < 20; ++k) bstate_cells[20 * (int64_t)L.cell_of_slot[s] + k] = bstate[20 * s + k];
    return 0;
}

// forward and backward prediction passes with the cooperative step, role by role, in the order of
// ggp_loglik_coop_kernel<.., PRED = true> and ggp_backward_coop_kernel (ggp_coop_kernels.cuh)
int hc_predict_coop(const ggp_forest_desc* d, const double* params, int n_seg, double* fwd, double* bwd, double* bstate_cells) {
    GgpLayout L;
    if (!L.build(d).empty() || L.max_seg >= n_seg) return -1;
    double scratch[GGP_CS_COUNT];
    const GgpScratch S{scratch, 1};
    const GgpDevForest F = hc_dev(L, d);
    std::vector<double> state((size_t)14 * L.n_cells), bstate((size_t)20 * L.n_cells);
    for (int64_t slot = 0; slot < L.n_cells; ++slot) {   // forward: generation order
        const int64_t off = F.s_off[slot];
        const int n = F.s_n[slot], parent = F.s_parent[slot];
        int t = 0;
        int64_t from = off;
        if (parent < 0) {
            double mu[4], C[16];
            ggp_root_start(mu, C, nullptr, F, params + GGP_NP * F.seg[off], off, &g_tables, [](double) {});
            ggp_store20(fwd + 20 * off, mu, C);
            GgpState s;
            ggp_state_from16(s, mu, C);
            for (int k = 0; k < 4; ++k) S[GGP_CS_ST + k] = s.m[k];
            for (int k = 0; k < 10; ++k) S[GGP_CS_ST + 4 + k] = s.c[k];
        } else {
            for (int k = 0; k < 14; ++k) S[GGP_CS_ST + k] = state[k * L.n_cells + parent];
            t = -1;
            from = F.s_off[parent] + F.s_n[parent] - 1;
        }
        while (t + 1 < n) {
            const int64_t at = off + t + 1;
            const double* p = params + GGP_NP * F.seg[from];
            const double* pt = params + GGP_NP * F.seg[at];
            const double dt = F.time[at] - F.time[from];
            for (int ph = 0; ph < GGP_COOP_PHASES; ++ph)
                for (int role = 0; role < GGP_COOP_ROLES; ++role) ggp_coop_run_phase(ph, role, S, ggp_ou(p, false), dt, &g_tables);
            for (int role = 0; role < GGP_COOP_ROLES; ++role)
                ggp_coop_ph3_pred<false>(role, S, t < 0, p, pt, F.x[at], F.g[at], F.model, &g_tables, fwd + 20 * at);
            ++t;
            from = at;
        }
        for (int k = 0; k < 14; ++k) state[k * L.n_cells + slot] = S[GGP_CS_ST + k];
    }
    for (int64_t slot = L.n_cells - 1; slot >= 0; --slot) {   // backward: leaves first
        const int64_t off = F.s_off[slot];
        const int n = F.s_n[slot], d1 = F.s_d1[slot], d2 = F.s_d2[slot];
        const bool leaf = d1 < 0 && d2 < 0;
        const int da = d1 >= 0 ? d1 : d2;
        int t = leaf ? n - 1 : n;
        int64_t from = leaf ? off + t : F.s_off[da];
        const double* p0 = params + GGP_NP * F.seg[off + n - 1];
        double mu[4], C[16];
        if (leaf) {
            ggp_leaf_start(mu, C, F, fwd, bwd, p0, from);
            if (t == 0) ggp_store20(bstate.data() + 20 * slot, mu, C);
        } else {
            ggp_mother_start(mu, C, bstate.data(), d1, d2, p0, F.model);
        }
        GgpState s;
        ggp_state_from16(s, mu, C);
        for (int k = 0; k < 4; ++k) S[GGP_CS_ST + k] = s.m[k];
        for (int k = 0; k < 10; ++k) S[GGP_CS_ST + 4 + k] = s.c[k];
        while (t > 0) {
            const int64_t at = off + t - 1;
            const double* pp = params + GGP_NP * F.seg[at];
            const double dt = F.time[from] - F.time[at];
            for (int ph = 0; ph < GGP_COOP_PHASES; ++ph)
                for (int role = 0; role < GGP_COOP_ROLES; ++role) ggp_coop_run_phase(ph, role, S, ggp_ou(pp, true), dt, &g_tables);
            for (int role = 0; role < GGP_COOP_ROLES; ++role) ggp_coop_store_reversed(role, S, bwd + 20 * at);
            --t;
            for (int role = 0; role < GGP_COOP_ROLES; ++role)
                ggp_coop_ph3_pred<false>(role, S, false, pp, pp, F.x[at], F.g[at], F.model, &g_tables, t == 0 ? bstate.data() + 20 * slot : nullptr);
            from = at;
        }
    }
    for (int64_t s = 0; s < L.n_cells; ++s)
        for (int k = 0; k < 20; ++k) bstate_cells[20 * (int64_t)L.cell_of_slot[s] + k] = bstate[20 * s + k];
    return 0;
}

// joints on the host: predict, per-ctp preparation, then one walker over every start point (row), rows in ctp order;
// returns the number of joints, writes at most cap (unsorted inside a row: emission order)
long long hc_joints(const ggp_forest_desc* d, const double* params, int n_seg, double tol, long long cap, long long* row, long long* col, double* rec44) {
    GgpLayout L;
    if (!L.build(d).empty() || L.max_seg >= n_seg) return -1;
    double scratch[GGP_SCRATCH];
    const GgpScratch S{scratch, 1};
    const GgpDevForest F = hc_dev(L, d);
    std::vector<double> state((size_t)14 * L.n_cells), bstate((size_t)20 * L.n_cells), fwd((size_t)20 * L.n_ctp), bwd((size_t)20 * L.n_ctp);
    GgpFwdArgs A{};
    A.params = params; A.v_count = 1; A.state = state.data(); A.out_fwd = fwd.data();
    for (int64_t s = 0; s < L.n_cells; ++s) ggp_cell_forward<true, false>(F, A, (int)s, 0, nullptr, &g_tables, S, nullptr);
    GgpBwdArgs B{};
    B.params = params; B.fwd = fwd.data(); B.bwd = bwd.data(); B.bstate = bstate.data();
    for (int64_t s = L.n_cells - 1; s >= 0; --s) ggp_cell_backward(F, B, (int)s, &g_tables, S);
    std::vector<double> prep((size_t)GGP_JOINT_PREP * L.n_ctp), stack((size_t)72 * (L.n_gen + 1));
    std::vector<int32_t> stack_slot(L.n_gen + 1);
    unsigned long long count = 0, next_row = 0;
    GgpJointArgs J{};
    J.params = params; J.fwd = fwd.data(); J.bwd = bwd.data(); J.bstate = bstate.data(); J.prep = prep.data();
    J.ctp_slot = L.ctp_slot.data(); J.tol = tol; J.cap = cap; J.count = &count; J.row_ctp = row; J.col_ctp = col; J.rec44 = rec44;
    J.stack = stack.data(); J.stack_slot = stack_slot.data(); J.stack_depth = L.n_gen + 1;
    for (int64_t k = 0; k < L.n_ctp; ++k) ggp_ctp_joint_prep(F, J, k, &g_tables, S);
    J.next_row = &next_row; J.row_begin = 0; J.row_end = L.n_ctp;
    ggp_walk_start_points(F, J, 0);   // one walker takes every start point in turn
    return (long long)count;
}
}
