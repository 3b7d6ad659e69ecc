// tests/hostcheck/simcheck.cpp — the simulator of ggp_sim.cuh compiled for the host (g++ -ffp-contract=off): the device
// kernel's per-cell body driven over the slots in generation order, as ggp_simulate launches it, so a CPU build returns the
// device's bits.  Test infrastructure (tests/test_sim_host.py, tests/test_gpu_sim.py, tools/sim_check.py); not part of the product.
#include <vector>

#include "../../gfp_gaussian_process_b200/csrc/ggp_tables_data.h"
#include "../../gfp_gaussian_process_b200/csrc/ggp_layout.hpp"
#include "../../gfp_gaussian_process_b200/csrc/ggp_sim.cuh"

static const GgpMathTables g_tables = GGP_MATH_TABLES_INIT;

extern "C" {
// Philox4x32-10 of one counter: out [4]
void sc_philox(const uint32_t* ctr, uint64_t key, uint32_t* out) { ggp_philox4x32_10(ctr, key, out); }

// the simulated series of the descriptor's forest: out_x, out_g [n_ctp] (caller's order); root4 NULL = the forest's init_f;
// *bad_cell = the first cell with a non-finite observation, -1 if none.  Returns 0, or -1 for a descriptor the library refuses
int sc_simulate(const ggp_forest_desc* d, const double* params, uint64_t seed, int substeps, const double* root4, double* out_x,
                double* out_g, long long* bad_cell) {
    GgpLayout L;
    if (!L.build(d).empty()) return -1;
    GgpDevForest F{};
    F.n_cells = L.n_cells; F.n_ctp = L.n_ctp;
    F.time = d->time; F.seg = L.seg.data();
    F.s_off = L.s_off.data(); F.s_n = L.s_n.data(); F.s_parent = L.s_parent.data(); F.s_d1 = L.s_d1.data();
    F.s_d2 = L.s_d2.data(); F.s_root = L.s_root.data(); F.s_cell = L.s_cell.data(); F.s_dfs0 = L.s_dfs0.data();
    F.model.noise_scaled = d->noise_model == GGP_NOISE_SCALED;
    F.model.division_binomial = d->division_model == GGP_DIVISION_BINOMIAL;
    F.model.fp_auto = d->fp_auto;
    std::vector<double> end((size_t)L.n_cells * 4), edge((size_t)L.n_cells * 4);
    unsigned long long bad = ~0ull;
    GgpSimArgs A{};
    A.params = params;
    for (int i = 0; i < 4; ++i) A.root[i] = root4 ? root4[i] : L.init_f[i];
    A.seed = seed;
    A.substeps = substeps;
    A.key = nullptr;
    A.end = end.data();
    A.edge = edge.data();
    A.bad_key = &bad;
    A.x_out = out_x;
    A.g_out = out_g;
    for (int64_t slot = 0; slot < L.n_cells; ++slot) ggp_sim_cell(F, A, (int)slot, &g_tables);
    *bad_cell = bad == ~0ull ? -1 : (long long)bad;
    return 0;
}
}
