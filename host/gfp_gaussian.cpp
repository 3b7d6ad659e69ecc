// host/gfp_gaussian.cpp — the `gfp_gaussian` command line on top of libggp_b200.so.
//
// Same options, input formats, running modes, output files and log-file life cycle as the reference's main.cpp
// (arg_parser :191-330, main :340-464, run_minimization :23-74, run_bound_1dscan :77-112,
// run_prediction_segments :115-147, run_joint_distribution :150-186) and the writers of likelihood.h:125-159,
// :275-377, predictions.h:505-601 and correlation_tree.h:96-126, :588-648, :785-790 — so the build is a drop-in.
// Everything numerical is done on the GPU through the C ABI (include/ggp_b200.h); there is no CPU path: without a
// CUDA device the first mode that needs numbers fails with the library's error.
//
// What differs from the reference on purpose:
//   * parents are resolved with a hash map and the table is SoA (ggp_data.hpp), so large inputs load;
//   * a 1-d scan, the Hessian stencil (1 200 evaluations for the example) and the simplex start/shrink are single
//     batched launches; results are those of one-by-one evaluation (the library chains the reference's history
//     dependence, SURVEY.md H3, through `root_carry` in evaluation order);
//   * NLopt is replaced by ggp_neldermead.hpp (iterate parity unpinned);
//   * extra options: --device N, --devices a,b,.. (lineage trees sharded over several GPUs behind one library handle, ggp_group:
//     likelihood, predictions, joints and correlation sums all run on every device), --fresh (every evaluation starts from zero root off-diagonals, i.e. is a pure
//     function of the parameters; enables speculative batching of the simplex moves), --sparse_joints (one line per
//     joint instead of the dense matrix whose size is quadratic in the data set).
#include <cstdio>
#include <cstring>
#include <filesystem>
#include <fstream>
#include <iomanip>
#include <iostream>
#include <memory>
#include <thread>

#include "ggp_correlation.hpp"
#include "ggp_data.hpp"
#include "ggp_neldermead.hpp"
#include "ggp_params.hpp"

using namespace ggp;

namespace {

struct Session {
    Args args;
    std::ofstream log;
    int print_level = 0;
    int iteration = 0;        // likelihood.h:7
    bool save_ll = false;     // likelihood.h:9
    std::ofstream file_iteration;
    std::vector<int> devices{0};   // --devices: trees are sharded over these (one forest handle per device)
    bool fresh = false;
};

void check(int rc, const char* what) {
    if (rc != GGP_OK) throw std::runtime_error(std::string(what) + ": " + ggp_last_error());
}

// what the running modes need from "the data on the GPU(s)"
class Forest {
public:
    virtual ~Forest() = default;
    virtual const LineageTable& table() const = 0;
    // +log-likelihood of each vector, evaluated as if one after the other (likelihood.h:170-174)
    // tolerate_nan: a NaN evaluation is returned as NaN instead of being reported (speculative batches: the search may never
    // use that point; if it does, the point is evaluated again on its own and reported like the reference does)
    virtual std::vector<double> loglik(Session& S, const std::vector<std::vector<double>>& P, bool tolerate_nan = false) = 0;
    // combined predictions [n_ctp][20] in the table's ctp order (main.cpp:132-140)
    virtual void predict(const std::vector<double>& P, int n_seg, std::vector<double>& comb) = 0;
    // joints of the start points [r0, r1) in (row, col) order and the lag-binned correlation sums, in the table's ctp indices
    // (ggp_joints / ggp_correlation_sums; predict() with the same parameters comes first).  Return the library's status code.
    virtual int joints(const std::vector<double>& P, int n_seg, double tol, int64_t r0, int64_t r1, int64_t cap, int64_t* n,
                       int64_t* row, int64_t* col, double* rec) = 0;
    virtual int correlation_sums(const std::vector<double>& P, int n_seg, double tol, double step, int n_bins, double atol,
                                 bool normalize_time, double* hi, double* lo, int64_t* n_joints) = 0;
    // value, gradient [n] and Hessian [n][n] of the fast log-likelihood at p over the parameter indices dirs (ggp_loglik_hess)
    virtual int loglik_hess(const std::vector<double>& p, const std::vector<int32_t>& dirs, double* ll, double* grad, double* hess) = 0;
};

struct LoglikResult {
    int rc = GGP_OK;
    std::vector<double> ll;
    std::vector<ggp_nan_info> nan;
    std::string error;
};

[[noreturn]] void report_nan(Session& S, const LineageTable& T, int64_t cell, int64_t t_index, const std::vector<double>& p) {
    S.log << "(sc_likelihood) ERROR: Log likelihood is Nan\n_____________________________\nCell: " << T.cell_id[cell]
          << ", observation: " << t_index << "\nParameters:";
    for (double x : p) S.log << " " << std::setprecision(15) << x;
    S.log << "\n";
    throw std::domain_error("Likelihood is Nan");
}

// --fast: likelihood evaluations of -m / -s use the library's fast arithmetic (GGP_MODE_FAST: quadrature + FMA, within 1e-10 of
// the reference's log-likelihood, not bit-identical); implies --fresh, predictions and joints stay strict
static bool g_fast_likelihood = false;

// one data slice on one device + the roots' persistent covariance (the reference's MOMAdata::cov of the roots)
class DeviceForest : public Forest {
public:
    // init_f / init_r: the init_cells statistics to use (nullptr: those of this table, as init_cells(cells) computes them)
    DeviceForest(const LineageTable& T, int device, const double* init_f = nullptr, const double* init_r = nullptr) : table_(T) {
        ggp_forest_desc d = make_desc(T, device);
        if (init_f && init_r) {
            d.compute_init = 0;
            for (int i = 0; i < 4; ++i) { d.init_f[i] = init_f[i]; d.init_r[i] = init_r[i]; }
        }
        check(ggp_forest_create(&d, &h_), "ggp_forest_create");
        if (g_fast_likelihood) check(ggp_forest_set_mode(h_, GGP_MODE_FAST), "ggp_forest_set_mode");
        carry_.assign((size_t)ggp_forest_n_roots(h_) * 16, 0.0);
    }
    ~DeviceForest() override { ggp_forest_destroy(h_); }
    DeviceForest(const DeviceForest&) = delete;
    ggp_forest* handle() const { return h_; }
    const LineageTable& table() const override { return table_; }
    int joints(const std::vector<double>& P, int n_seg, double tol, int64_t r0, int64_t r1, int64_t cap, int64_t* n, int64_t* row,
               int64_t* col, double* rec) override {
        return ggp_joints(h_, P.data(), n_seg, tol, r0, r1, cap, n, row, col, rec);
    }
    int correlation_sums(const std::vector<double>& P, int n_seg, double tol, double step, int n_bins, double atol, bool normalize_time,
                         double* hi, double* lo, int64_t* n_joints) override {
        return ggp_correlation_sums(h_, P.data(), n_seg, tol, step, n_bins, atol, normalize_time ? 1 : 0, hi, lo, n_joints);
    }
    int loglik_hess(const std::vector<double>& p, const std::vector<int32_t>& dirs, double* ll, double* grad, double* hess) override {
        return ggp_loglik_hess(h_, p.data(), 1, dirs.data(), (int32_t)dirs.size(), ll, grad, hess, nullptr);
    }

    LoglikResult loglik_raw(const std::vector<double>& flat, int n_vec, bool fresh) {
        LoglikResult R;
        R.ll.resize(n_vec);
        R.nan.resize(n_vec);
        R.rc = ggp_loglik(h_, flat.data(), n_vec, fresh ? nullptr : carry_.data(), R.ll.data(), nullptr, R.nan.data());
        if (R.rc != GGP_OK && R.rc != GGP_ERR_NAN) R.error = ggp_last_error();
        return R;
    }
    std::vector<double> loglik(Session& S, const std::vector<std::vector<double>>& P, bool tolerate_nan = false) override {
        std::vector<double> flat;
        for (const auto& p : P) flat.insert(flat.end(), p.begin(), p.end());
        LoglikResult R = loglik_raw(flat, (int)P.size(), S.fresh);
        if (R.rc == GGP_ERR_NAN) {
            if (tolerate_nan) return R.ll;
            for (size_t v = 0; v < P.size(); ++v)
                if (R.nan[v].cell >= 0) report_nan(S, table_, R.nan[v].cell, R.nan[v].t_index, P[v]);
        }
        if (R.rc != GGP_OK) throw std::runtime_error("ggp_loglik: " + R.error);
        return R.ll;
    }
    void predict(const std::vector<double>& P, int n_seg, std::vector<double>& comb) override {
        comb.resize((size_t)table_.n_ctp() * 20);
        check(ggp_predict(h_, P.data(), n_seg, nullptr, nullptr, comb.data()), "ggp_predict");
    }

private:
    const LineageTable& table_;
    ggp_forest* h_ = nullptr;
    std::vector<double> carry_;
};

// The table's trees sharded over several devices behind ONE library handle (ggp_group, SURVEY.md 8b / 8e): every descendant
// stays with its root, the init_cells statistics are those of the whole table, one host thread per device inside a call; the
// per-shard log-likelihoods are added in shard order, prediction rows, joints and the first NaN come back in the table's order.
class GroupForest : public Forest {
public:
    GroupForest(const LineageTable& T, const std::vector<int>& devices) : table_(T) {
        const ggp_forest_desc d = make_desc(T, devices[0]);
        std::vector<int32_t> dev(devices.begin(), devices.end());
        check(ggp_group_create(&d, dev.data(), (int32_t)dev.size(), &g_), "ggp_group_create");
        if (g_fast_likelihood) check(ggp_group_set_mode(g_, GGP_MODE_FAST), "ggp_group_set_mode");
        int64_t n_roots = 0;
        for (int64_t c = 0; c < T.n_cells(); ++c) n_roots += T.parent[c] < 0;
        carry_.assign((size_t)n_roots * 16, 0.0);
    }
    ~GroupForest() override { ggp_group_destroy(g_); }
    GroupForest(const GroupForest&) = delete;
    const LineageTable& table() const override { return table_; }

    std::vector<double> loglik(Session& S, const std::vector<std::vector<double>>& P, bool tolerate_nan = false) override {
        std::vector<double> flat;
        for (const auto& p : P) flat.insert(flat.end(), p.begin(), p.end());
        const int n_vec = (int)P.size();
        std::vector<double> ll(n_vec);
        std::vector<ggp_nan_info> nan(n_vec);
        const int rc = ggp_group_loglik(g_, flat.data(), n_vec, S.fresh ? nullptr : carry_.data(), ll.data(), nullptr, nan.data());
        if (rc == GGP_ERR_NAN) {
            if (tolerate_nan) return ll;
            for (int v = 0; v < n_vec; ++v)
                if (nan[v].cell >= 0) report_nan(S, table_, nan[v].cell, nan[v].t_index, P[v]);
        }
        check(rc, "ggp_group_loglik");
        return ll;
    }
    void predict(const std::vector<double>& P, int n_seg, std::vector<double>& comb) override {
        comb.resize((size_t)table_.n_ctp() * 20);
        check(ggp_group_predict(g_, P.data(), n_seg, nullptr, nullptr, comb.data()), "ggp_group_predict");
    }
    int joints(const std::vector<double>& P, int n_seg, double tol, int64_t r0, int64_t r1, int64_t cap, int64_t* n, int64_t* row,
               int64_t* col, double* rec) override {
        return ggp_group_joints(g_, P.data(), n_seg, tol, r0, r1, cap, n, row, col, rec);
    }
    int correlation_sums(const std::vector<double>& P, int n_seg, double tol, double step, int n_bins, double atol, bool normalize_time,
                         double* hi, double* lo, int64_t* n_joints) override {
        return ggp_group_correlation_sums(g_, P.data(), n_seg, tol, step, n_bins, atol, normalize_time ? 1 : 0, hi, lo, n_joints);
    }
    int loglik_hess(const std::vector<double>& p, const std::vector<int32_t>& dirs, double* ll, double* grad, double* hess) override {
        return ggp_group_loglik_hess(g_, p.data(), 1, dirs.data(), (int32_t)dirs.size(), ll, grad, hess, nullptr);
    }

private:
    const LineageTable& table_;
    ggp_group* g_ = nullptr;
    std::vector<double> carry_;   // the roots' persistent covariance in the table's root order
};

std::unique_ptr<Forest> make_forest(Session& S, const LineageTable& T) {
    if (S.devices.size() > 1) return std::unique_ptr<Forest>(new GroupForest(T, S.devices));
    return std::unique_ptr<Forest>(new DeviceForest(T, S.devices[0]));
}

// bookkeeping of one evaluation (likelihood.h:138-158): counter, iterations file, stdout
void record_evaluation(Session& S, const std::vector<double>& p, double tl) {
    ++S.iteration;
    if (S.save_ll) {
        S.file_iteration << S.iteration << ",";
        for (double x : p) S.file_iteration << std::setprecision(20) << x << ",";
        S.file_iteration << std::setprecision(30) << tl << std::setprecision(15) << "\n";
    }
    if (S.print_level > 0) {
        std::cout << S.iteration << ": ";
        for (double x : p) std::cout << std::setprecision(20) << x << ", ";
        std::cout << "ll=" << std::setprecision(30) << tl << std::setprecision(15) << "\n";
    }
}

std::vector<double> total_likelihood(Session& S, Forest& F, const std::vector<std::vector<double>>& P, bool record = true) {
    std::vector<double> ll = F.loglik(S, P, /*tolerate_nan=*/!record);
    if (record) for (size_t v = 0; v < P.size(); ++v) record_evaluation(S, P[v], ll[v]);
    return ll;
}

void setup_outfile_likelihood(const std::string& outfile, const ParameterSet& params) {
    params.to_csv(outfile);
    std::ofstream f(outfile, std::ios_base::app);
    f << "\nlog_likelihoods:\niteration,";
    for (const Parameter& p : params.all) f << p.name << ",";
    f << "log_likelihood\n";
}

// ---- dense inverse by partially pivoted LU (what Eigen's MatrixXd::inverse() does; likelihood.h:262) ----
std::vector<double> invert(std::vector<double> A, int n) {
    std::vector<double> R((size_t)n * n, 0.0);
    std::vector<int> perm(n);
    for (int i = 0; i < n; ++i) perm[i] = i;
    for (int k = 0; k < n; ++k) {
        int piv = k;
        for (int i = k + 1; i < n; ++i) if (std::fabs(A[i * n + k]) > std::fabs(A[piv * n + k])) piv = i;
        if (piv != k) {
            for (int j = 0; j < n; ++j) std::swap(A[k * n + j], A[piv * n + j]);
            std::swap(perm[k], perm[piv]);
        }
        for (int i = k + 1; i < n; ++i) {
            A[i * n + k] /= A[k * n + k];
            for (int j = k + 1; j < n; ++j) A[i * n + j] -= A[i * n + k] * A[k * n + j];
        }
    }
    for (int c = 0; c < n; ++c) {
        std::vector<double> y(n);
        for (int i = 0; i < n; ++i) {
            double s = perm[i] == c ? 1.0 : 0.0;
            for (int j = 0; j < i; ++j) s -= A[i * n + j] * y[j];
            y[i] = s;
        }
        for (int i = n - 1; i >= 0; --i) {
            double s = y[i];
            for (int j = i + 1; j < n; ++j) s -= A[i * n + j] * R[j * n + c];
            R[i * n + c] = s / A[i * n + i];
        }
    }
    return R;
}

// squared error bars from the numerical Hessian (likelihood.h:211-269), the whole stencil in one launch
std::vector<double> ll_error_bars(Session& S, Forest& F, const ParameterSet& params, double epsilon) {
    const std::vector<double> x = params.get_final();
    const std::vector<int> idx = params.non_fixed();
    const int n = (int)idx.size();
    std::vector<std::vector<double>> P;
    std::vector<double> h1s, h2s;
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            const int ii = idx[i], jj = idx[j];
            const double h1 = std::max(x[ii] * epsilon, 1e-12), h2 = std::max(x[jj] * epsilon, 1e-12);
            for (int s = 0; s < 4; ++s) {
                std::vector<double> v = x;
                v[ii] = v[ii] + ((s & 2) ? -h1 : h1);
                v[jj] = v[jj] + ((s & 1) ? -h2 : h2);
                P.push_back(v);
            }
            h1s.push_back(h1); h2s.push_back(h2);
        }
    const std::vector<double> ll = total_likelihood(S, F, P);
    std::vector<double> H((size_t)n * n);
    for (int k = 0; k < n * n; ++k) H[k] = (ll[4 * k] - ll[4 * k + 1] - ll[4 * k + 2] + ll[4 * k + 3]) / (4 * h1s[k] * h2s[k]);
    const std::vector<double> Hi = invert(H, n);
    std::vector<double> err;
    for (int i = 0; i < n; ++i) err.push_back(-Hi[i * n + i]);
    return err;
}

void save_error_bars(Session& S, Forest& F, const std::string& outfile, const ParameterSet& params) {
    std::ofstream f(outfile, std::ios_base::app);
    f << "\nerrors^2:\nepsilon";
    const std::vector<int> idx = params.non_fixed();
    for (int i : idx) f << "," << params.all[i].name;
    f << "\n";
    for (double eps : {5e-2, 1e-2, 5e-3}) {
        const std::vector<double> e = ll_error_bars(S, F, params, eps);
        f << eps;
        for (double v : e) f << "," << v;
        f << "\n";
    }
}

// --exact_errors: squared error bars -diag(H^-1) from the exact Hessian of the fast log-likelihood over the free parameters at
// the final parameters (ggp_loglik_hess, natural space): one row, no step size
void save_exact_error_bars(Forest& F, const std::string& outfile, const ParameterSet& params) {
    const std::vector<int> idx = params.non_fixed();
    const int n = (int)idx.size();
    if (n == 0) return;
    const std::vector<int32_t> dirs(idx.begin(), idx.end());
    double ll = 0.0;
    std::vector<double> grad(n), H((size_t)n * n);
    check(F.loglik_hess(params.get_final(), dirs, &ll, grad.data(), H.data()), "ggp_loglik_hess");
    const std::vector<double> Hi = invert(H, n);
    std::ofstream f(outfile, std::ios_base::app);
    f << "\nerrors^2 (exact Hessian of the fast log-likelihood):\n";
    for (int i = 0; i < n; ++i) f << (i ? "," : "") << params.all[idx[i]].name;
    f << "\n" << std::setprecision(17);
    for (int i = 0; i < n; ++i) f << (i ? "," : "") << -Hi[(size_t)i * n + i];
    f << "\n";
}

void save_final_likelihood(const std::string& outfile, const LineageTable& T, double ll_max, double tolerance, Args& a) {
    std::ofstream f(outfile, std::ios_base::app);
    const long n = (long)T.n_ctp();
    f << "\nn_data_points, " << n << "\n";
    f << "total_log_likelihoood," << std::setprecision(15) << ll_max << "\n";
    f << "norm_log_likelihoood," << std::setprecision(15) << ll_max / n << "\n";
    f << "optimization_algorithm,LN_NELDERMEAD\n";
    f << "tolerance," << tolerance << "\n";
    f << "search_space," << a["search_space"] << "\n";
    f << "noise_model," << a["noise_model"] << "\n";
    f << "cell_division_model," << a["cell_division_model"] << "\n";
    f << "version,0.4.2-ggp-b200\n";
}

// ---- running modes ---------------------------------------------------------------------------------
void run_minimization(Session& S, const LineageTable& T, ParameterSet& params, int segment) {
    S.log << "-> Minimizaton\n";
    const std::string base = out_dir(S.args) + with_segment(file_base(S.args["infile"]), segment) + params.code();
    const std::string outfile_ll = base + "_iterations.csv";
    S.file_iteration = std::ofstream(outfile_ll, std::ios_base::app);
    setup_outfile_likelihood(outfile_ll, params);
    S.log << "Outfile: " << outfile_ll << "\n";

    const std::unique_ptr<Forest> Fp = make_forest(S, T);
    Forest& F = *Fp;
    const bool log_space = S.args["search_space"] == "log";
    const double tolerance = std::stod(S.args["tolerance_maximization"]);
    const size_t n = params.all.size();
    std::vector<double> x(n), lb(n), ub(n), step(n);
    for (size_t i = 0; i < n; ++i) {
        const Parameter& p = params.all[i];
        const double start = p.minimized ? p.final_value : p.init;
        x[i] = log_space ? std::log(start) : start;
        if (p.fixed) {
            step[i] = 1.;
            lb[i] = ub[i] = log_space ? std::log(p.init) : p.init;
        } else {
            step[i] = log_space ? std::log(1. + p.step / p.init) : p.step;
            lb[i] = log_space ? std::log(p.lower) : p.lower;
            ub[i] = log_space ? std::log(p.upper) : p.upper;
        }
    }
    auto natural = [&](const std::vector<double>& y) {
        std::vector<double> p = y;
        if (log_space) for (double& v : p) v = std::exp(v);
        return p;
    };
    BatchObjective obj;
    obj.evaluate = [&](const std::vector<std::vector<double>>& Y, bool record) {
        std::vector<std::vector<double>> P;
        for (const auto& y : Y) P.push_back(natural(y));
        std::vector<double> ll = total_likelihood(S, F, P, record);
        for (double& v : ll) v = -v;
        return ll;
    };
    obj.commit = [&](const std::vector<double>& y, double f) { record_evaluation(S, natural(y), -f); };
    S.save_ll = true;
    S.log << "Optimization algorithm: Nelder-Mead simplex (bounded, batched) Tolerance: " << tolerance << "\n";
    S.iteration = 0;
    // how many parameter vectors a speculative launch may hold: a launch over a small data set is a chain of dependent steps that
    // costs the same for 1 or 200 vectors, over a large one every vector costs its share (4 = this iteration's candidates only)
    int spec_batch = (int)std::min<int64_t>(192, std::max<int64_t>(4, (int64_t)4000000 / std::max<int64_t>(1, T.n_ctp())));
    if (const char* m = getenv("GGP_B200_SPEC_BATCH")) spec_batch = std::max(1, atoi(m));
    const NelderMeadResult R = nelder_mead(obj, x, lb, ub, step, tolerance, /*speculate=*/S.fresh, 0, spec_batch);
    S.save_ll = false;
    const double ll_max = -R.f;
    S.log << "Stopped: " << R.reason << " after " << R.evaluations << " evaluations in " << R.launches << " launches\n";
    S.log << "Found maximum: log likelihood = " << std::setprecision(20) << ll_max << std::setprecision(10) << "\n";
    params.set_final(natural(R.x));
    S.log << params << std::endl;
    S.file_iteration.close();

    S.log << "-> Error estimation\n";
    const std::string outfile_final = base + "_final.csv";
    S.log << "Outfile: " << outfile_final << "\n";
    params.to_csv(outfile_final);
    save_error_bars(S, F, outfile_final, params);
    save_final_likelihood(outfile_final, T, ll_max, tolerance, S.args);
    if (S.args.count("exact_errors")) save_exact_error_bars(F, outfile_final, params);

    std::ofstream pf(base + "_parameter_file.txt");
    pf << "# Generated parameter file with the final parameters that may be used for predictions\n";
    for (const Parameter& p : params.all) pf << p.name << " = " << p.final_value << "\n";
}

void run_bound_1dscan(Session& S, const LineageTable& T, const ParameterSet& params, int segment) {
    S.log << "-> 1d Scan\n";
    const std::unique_ptr<Forest> Fp = make_forest(S, T);
    Forest& F = *Fp;
    S.save_ll = true;
    for (size_t i = 0; i < params.all.size(); ++i) {
        const Parameter& p = params.all[i];
        if (!p.bound) continue;
        const std::string outfile = out_dir(S.args) + with_segment(file_base(S.args["infile"]), segment) + "_scan_" + p.name + ".csv";
        S.file_iteration = std::ofstream(outfile, std::ios_base::app);
        setup_outfile_likelihood(outfile, params);
        S.log << "Outfile: " << outfile << "\n";
        std::vector<std::vector<double>> P;
        for (double v : arange(p.lower, p.upper, p.step)) {
            P.push_back(params.get_final());
            P.back()[i] = v;
        }
        if (!P.empty()) total_likelihood(S, F, P);   // all samples of this parameter in one launch
        S.file_iteration.close();
    }
    S.save_ll = false;
}

struct Predictions { std::vector<double> fwd, bwd, comb; };

std::vector<double> flatten_params(const std::vector<ParameterSet>& list) {
    std::vector<double> P;
    for (const ParameterSet& ps : list) { const auto v = ps.get_final(); P.insert(P.end(), v.begin(), v.end()); }
    return P;
}

std::string prediction_base(Session& S, const std::vector<ParameterSet>& list) {
    std::string f = out_dir(S.args) + file_base(S.args["infile"]);
    for (const ParameterSet& ps : list) f += ps.code();
    return f;
}

void run_prediction_segments(Session& S, Forest& F, std::vector<ParameterSet>& list) {
    S.log << "-> prediction\n";
    const LineageTable& T = F.table();
    const std::string outfile = prediction_base(S, list) + "_prediction.csv";
    const std::vector<double> P = flatten_params(list);
    std::vector<double> comb;
    F.predict(P, (int)list.size(), comb);
    S.log << "Outfile: " << outfile << "\n";
    for (size_t i = 0; i < list.size(); ++i) list[i].to_csv(outfile, i == 0 ? std::ios_base::out : std::ios_base::app);
    std::ofstream f(outfile, std::ios_base::app);
    f << "\ncell_id,parent_id,time,log_length,fp,mean_x,mean_g,mean_l,mean_q,cov_xx,cov_xg,cov_xl,cov_xq,cov_gg,cov_gl,cov_gq,cov_ll,cov_lq,cov_qq\n";
    for (int64_t c = 0; c < T.n_cells(); ++c)
        for (int64_t k = T.offset[c]; k < T.offset[c + 1]; ++k) {
            const double* r = comb.data() + 20 * k;
            f << T.cell_id[c] << "," << T.parent_id[c] << "," << T.time[k] << "," << T.log_length[k] << "," << T.fp[k] << ",";
            for (int i = 0; i < 4; ++i) f << (i ? "," : "") << r[i];
            for (int m = 0; m < 4; ++m)
                for (int n = m; n < 4; ++n) f << "," << r[4 + 4 * m + n];
            f << "\n";
        }
}

const int64_t kJointRowBlock = 32768;   // start points per ggp_joints call

// Records of the start points [r0, r1) in (row, col) order.  One library call when the buffers of the previous block
// were large enough (they grow with the densest block seen), otherwise a second one with the exact size.
void fetch_joints(Forest& Fx, const std::vector<double>& P, int n_seg, double tol, int64_t r0, int64_t r1,
                  std::vector<int64_t>& row, std::vector<int64_t>& col, std::vector<double>& rec, int64_t& n) {
    int64_t cap = (int64_t)std::min(row.size(), std::min(col.size(), rec.size() / 44));
    if (cap < 64 * (r1 - r0)) {
        cap = 64 * (r1 - r0);
        row.resize(cap); col.resize(cap); rec.resize((size_t)cap * 44);
    }
    check(Fx.joints(P, n_seg, tol, r0, r1, cap, &n, row.data(), col.data(), rec.data()), "ggp_joints");
    if (n > cap) {
        cap = n + n / 8;
        row.resize(cap); col.resize(cap); rec.resize((size_t)cap * 44);
        check(Fx.joints(P, n_seg, tol, r0, r1, cap, &n, row.data(), col.data(), rec.data()), "ggp_joints");
    }
}

void run_joint_distribution(Session& S, Forest& Fx, std::vector<ParameterSet>& list) {
    S.log << "-> joint posteriors\n";
    const LineageTable& T = Fx.table();
    // run_prediction_segments has left the predictions on the data set's handle(s); with several devices every shard walks its
    // own trees and the records come back in the table's row order (ggp_group_joints)
    const std::vector<double> P = flatten_params(list);
    const double tol = std::stod(S.args["rel_tolerance_joints"]);
    const bool sparse = S.args.count("sparse_joints") > 0;
    std::ofstream f(prediction_base(S, list) + "_joints.csv");
    for (const ParameterSet& ps : list) ps.to_csv(f);
    f << "\ncell_id,parent_id,time";
    const int64_t M = T.n_ctp();
    std::vector<int64_t> cell_of(M);
    for (int64_t c = 0; c < T.n_cells(); ++c) for (int64_t k = T.offset[c]; k < T.offset[c + 1]; ++k) cell_of[k] = c;
    if (sparse) {
        f << ",col_cell_id,col_time,joint(8 means + 36 upper-triangular covariances)\n";
    } else {   // dense header: one column block per cell-timepoint of the data set (correlation_tree.h:113-126, :640-642)
        f << ",";
        for (int64_t k = 0; k < M; ++k) f << T.cell_id[cell_of[k]] << '_' << T.time[k] << std::string(k == M - 1 ? 43 : 44, ',');
        f << "\n";
    }
    // rows are streamed in blocks like the reference streams lines (a block keeps every SM's walkers busy)
    const int64_t block = kJointRowBlock;
    std::vector<int64_t> row, col;
    std::vector<double> rec;
    for (int64_t r0 = 0; r0 < M; r0 += block) {
        const int64_t r1 = std::min(M, r0 + block);
        int64_t n = 0;
        fetch_joints(Fx, P, (int)list.size(), tol, r0, r1, row, col, rec, n);
        int64_t at = 0;
        for (int64_t r = r0; r < r1; ++r) {
            const int64_t c = cell_of[r];
            if (sparse) {
                for (; at < n && row[at] == r; ++at) {
                    f << T.cell_id[c] << "," << T.parent_id[c] << "," << T.time[r] << "," << T.cell_id[cell_of[col[at]]] << "," << T.time[col[at]];
                    for (int i = 0; i < 44; ++i) f << "," << rec[44 * at + i];
                    f << "\n";
                }
                continue;
            }
            f << T.cell_id[c] << "," << T.parent_id[c] << "," << T.time[r];
            int64_t next_col = 0;
            for (; at < n && row[at] == r; ++at) {
                f << std::string((size_t)(col[at] - next_col) * 44, ',');
                for (int i = 0; i < 44; ++i) f << "," << rec[44 * at + i];
                next_col = col[at] + 1;
            }
            f << std::string((size_t)(M - next_col) * 44, ',') << "\n";
        }
    }
}

// correlation functions (python_src/correlation_from_joint.py) from the joints on the device, no joints file in between
CorrelationSet make_correlation_set(Session& S) {
    const double dt = std::stod(S.args["correlation"]), n_data = std::stod(S.args["n_data"]);
    if (S.args.count("normalize_time")) return CorrelationSet(0.05, 3.0, 0.024);   // process_file :688-693
    return CorrelationSet(dt, dt * n_data, dt * 0.2);                              // :681-685
}

void run_correlation(Session& S, Forest& Fx, std::vector<ParameterSet>& list) {
    S.log << "-> correlation functions\n";
    const LineageTable& T = Fx.table();
    const std::vector<double> P = flatten_params(list);
    const double tol = std::stod(S.args["rel_tolerance_joints"]);
    std::vector<double> comb;
    CorrelationSet CS = make_correlation_set(S);
    // the lag-binned sums are accumulated on the device (ggp_correlation_sums: neither a joints file nor a record leaves the GPU);
    // the host reduction of the sparse records remains for what the device path refuses (parents stored after their daughters)
    // and for GGP_B200_CORR_HOST=1 (A/B comparison)
    bool on_device = false;
    if (!getenv("GGP_B200_CORR_HOST")) {
        // run_prediction_segments has left the predictions on the data set's own handle(s)
        std::vector<double> hi(CS.bins.size() * 50), lo(CS.bins.size() * 50);
        int64_t n_joints = 0;
        const double step = CS.bins.size() > 1 ? CS.bins[1].dt - CS.bins[0].dt : 1.0;
        const int rc = Fx.correlation_sums(P, (int)list.size(), tol, step, (int)CS.bins.size(), CS.tol,
                                           S.args.count("normalize_time") > 0, hi.data(), lo.data(), &n_joints);
        if (rc == GGP_OK) {
            CS.set_sums(hi.data(), lo.data());
            S.log << "   " << n_joints << " joints reduced into " << CS.bins.size() << " lag bins on the device\n";
            on_device = true;
        } else if (rc != GGP_ERR_BAD_ARG) {
            check(rc, "ggp_correlation_sums");
        } else {
            S.log << "   device reduction not applicable (" << ggp_last_error() << "): host reduction\n";
        }
    }
    if (!on_device) {
    Fx.predict(P, (int)list.size(), comb);
    std::vector<double> m14((size_t)T.n_ctp() * 14);
    for (int64_t k = 0; k < T.n_ctp(); ++k) {
        const double* r = comb.data() + 20 * k;
        double* o = m14.data() + 14 * k;
        for (int i = 0; i < 4; ++i) o[i] = r[i];
        int q = 4;
        for (int a = 0; a < 4; ++a) for (int b = a; b < 4; ++b) o[q++] = r[4 + 4 * a + b];
    }
    JointsSource src;
    src.marginal14 = [&](int64_t k) { return m14.data() + 14 * k; };
    src.joints_of_rows = [&](int64_t r0, int64_t r1, std::vector<int64_t>& row, std::vector<int64_t>& col, std::vector<double>& rec) {
        int64_t n = 0;
        row.resize(row.capacity()); col.resize(col.capacity());   // reuse what the previous block grew to
        fetch_joints(Fx, P, (int)list.size(), tol, r0, r1, row, col, rec, n);
        row.resize(n); col.resize(n);
    };
    correlation_from_joints(CS, T.cell_id, T.parent_id, T.offset, T.time, src, S.args.count("normalize_time") > 0, kJointRowBlock);
    }
    CS.finalize();
    const std::string outfile = prediction_base(S, list) + "_correlations.csv";
    S.log << "Outfile: " << outfile << "\n";
    CS.to_csv(outfile);
}

// ---- command line (main.cpp:191-330) ------------------------------------------------------------------
Args arg_parser(int argc, char** argv) {
    const std::vector<std::vector<std::string>> keys = {
        {"-h", "--help", "this help message"},
        {"-i", "--infile", "(required) input data file"},
        {"-b", "--parameter_bounds", "(required) file(s) setting the type, step, bounds of the parameters"},
        {"-c", "--csv_config", "file that sets the columns that will be used from the input file"},
        {"-l", "--print_level", "print level {0,1,2}, default: 0"},
        {"-o", "--outdir", "specify output direction and do not use default"},
        {"-t", "--tolerance_maximization", "absolute tolerance of maximization between optimization steps, default: 1e-10"},
        {"-r", "--rel_tolerance_joints", "relative tolerance of joint calculation: default 1e-10"},
        {"-space", "--search_space", "search parameter space in {'log'|'linear'} space, default: 'log'"},
        {"-noise", "--noise_model", "measurement noise of fp content {'scaled'|'const'} default: 'scaled'"},
        {"-div", "--cell_division_model", "cell divison model {'binomial'|'gauss'} default: 'binomial'"},
        {"-m", "--maximize", "run maximization"},
        {"-s", "--scan", "run 1d parameter scan"},
        {"-p", "--predict", "run prediction"},
        {"-j", "--joints", "run calculation of joint probabilities"},
        {"-d", "--device", "(ggp-b200) CUDA device ordinal, default: 0"},
        {"-ds", "--devices", "(ggp-b200) comma separated CUDA device ordinals: lineage trees are sharded over them"},
        {"-fresh", "--fresh", "(ggp-b200) history-free evaluations, speculative batching of simplex moves"},
        {"-fast", "--fast", "(ggp-b200) fast likelihood arithmetic for -m / -s (within 1e-10 of the reference, not bit-identical); implies --fresh"},
        {"-ee", "--exact_errors", "(ggp-b200) with -m: also the error bars of the exact Hessian of the fast log-likelihood (one more _final.csv section)"},
        {"-sj", "--sparse_joints", "(ggp-b200) write one line per joint instead of the dense matrix"},
        {"-corr", "--correlation", "(ggp-b200) time between measurements: correlation functions straight from the joints (implies -p; no joints file)"},
        {"-n_data", "--n_data", "(ggp-b200) number of lags of the correlation function, default: 200"},
        {"-norm", "--normalize_time", "(ggp-b200) correlation over time in units of the cell cycle"},
        {"-corr_files", "--correlation_files", "(ggp-b200) <prefix>_joints.csv: correlation functions from existing files (no GPU needed; use with -corr)"}};
    Args a;
    a["print_level"] = "0"; a["tolerance_maximization"] = "1e-10"; a["rel_tolerance_joints"] = "1e-10";
    a["search_space"] = "log"; a["noise_model"] = "scaled"; a["cell_division_model"] = "binomial"; a["device"] = "0"; a["n_data"] = "200";
    auto value = [&](int i) -> std::string {
        if (i + 1 >= argc) throw std::invalid_argument(std::string("missing value after ") + argv[i]);
        return argv[i + 1];
    };
    for (int i = 1; i < argc; ++i) {
        const std::string arg = argv[i];
        for (const auto& k : keys) {
            if (arg != k[0] && arg != k[1]) continue;
            const std::string& key = k[0];
            if (key == "-i") a["infile"] = value(i);
            else if (key == "-b") {
                std::string list;
                for (int j = i + 1; j < argc && std::string(argv[j]).rfind("-", 0) != 0; ++j) list += std::string(argv[j]) + " ";
                a["parameter_bounds"] = trim(list);
            } else if (key == "-c") a["csv_config"] = value(i);
            else if (key == "-l") a["print_level"] = value(i);
            else if (key == "-o") a["outdir"] = value(i);
            else if (key == "-t") a["tolerance_maximization"] = value(i);
            else if (key == "-r") a["rel_tolerance_joints"] = value(i);
            else if (key == "-space") a["search_space"] = value(i);
            else if (key == "-noise") a["noise_model"] = value(i);
            else if (key == "-div") a["cell_division_model"] = value(i);
            else if (key == "-m") a["minimize"] = "1";
            else if (key == "-s") a["scan"] = "1";
            else if (key == "-p") a["predict"] = "1";
            else if (key == "-j") { a["joints"] = "1"; a["predict"] = "1"; }
            else if (key == "-d") a["device"] = value(i);
            else if (key == "-ds") a["devices"] = value(i);
            else if (key == "-fresh") a["fresh"] = "1";
            else if (key == "-fast") { a["fast"] = "1"; a["fresh"] = "1"; }
            else if (key == "-ee") a["exact_errors"] = "1";
            else if (key == "-sj") a["sparse_joints"] = "1";
            else if (key == "-corr") { a["correlation"] = value(i); a["predict"] = "1"; }
            else if (key == "-n_data") a["n_data"] = value(i);
            else if (key == "-norm") a["normalize_time"] = "1";
            else if (key == "-corr_files") a["correlation_files"] = value(i);
            else if (key == "-h") {
                a["help"] = "1";
                std::cout << "Usage: ./gfp_gaussian [-options]\n";
                for (const auto& kk : keys) std::cout << pad(kk[0] + ", " + kk[1], 35) << kk[2] << "\n";
            }
        }
    }
    if (a.count("help")) return a;
    auto bad = [](const std::string& msg) { std::cout << "(arg_parser) ERROR: " << msg; throw std::invalid_argument("Invalide argument"); };
    if (a["search_space"] != "log" && a["search_space"] != "linear") bad("search_space must be either 'log' or 'linear', not " + a["search_space"]);
    if (a["noise_model"] != "const" && a["noise_model"] != "scaled") bad("noise_model must be either 'const' or 'scaled', not " + a["noise_model"]);
    if (a["cell_division_model"] != "gauss" && a["cell_division_model"] != "binomial")
        bad("cell_division_model must be either 'gauss' or 'binomial', not " + a["cell_division_model"]);
    if (a.count("correlation_files") && !a.count("infile")) a["infile"] = a["correlation_files"];
    if (!a.count("infile")) bad("Required infile flag not set!\n");
    if (!std::filesystem::exists(a["infile"])) bad("Infile " + a["infile"] + " not found (use '-h' for help)!\n");
    if (a.count("correlation_files")) return a;
    if (!a.count("parameter_bounds") || a["parameter_bounds"].empty()) bad("Required parameter_bounds flag not set!\n");
    for (const auto& pf : split(a["parameter_bounds"], " "))
        if (!std::filesystem::exists(pf)) bad("Paramters bound file '" + pf + "' not found (use '-h' for help)!\n");
    if (a.count("csv_config") && !std::filesystem::exists(a["csv_config"]))
        bad("csv_config flag set, but csv configuration file " + a["csv_config"] + " not found!\n");
    return a;
}

}  // namespace

int main(int argc, char** argv) {
    std::string outfile_log, outfile_log_success, outfile_log_error;
    Session S;
    std::cout << "Running... \n";
    try {
        S.args = arg_parser(argc, argv);
        if (S.args.count("help")) return EXIT_SUCCESS;
        S.print_level = std::stoi(S.args["print_level"]);
        S.devices.clear();
        for (const auto& d : split(S.args.count("devices") ? S.args["devices"] : S.args["device"], ",")) S.devices.push_back(std::stoi(trim(d)));
        S.fresh = S.args.count("fresh") > 0;
        g_fast_likelihood = S.args.count("fast") > 0;
        const std::string log_base = out_dir(S.args) + file_base(S.args["infile"]);
        outfile_log = log_base + ".log";
        outfile_log_success = log_base + "_success.log";
        outfile_log_error = log_base + "_error.log";
        S.log = std::ofstream(outfile_log, std::ios_base::app);
        std::cout << "Temporary log file '" << outfile_log << "' created\n";
        S.log << ggp_version() << "\n";

        if (S.args.count("correlation_files")) {   // drop-in for correlation_from_joint.py on existing files
            if (!S.args.count("correlation")) throw std::invalid_argument("--correlation_files needs --correlation <dt>");
            const std::string jf = S.args["correlation_files"];
            const size_t at = jf.rfind("joints");
            if (at == std::string::npos) throw std::invalid_argument("--correlation_files: not a <prefix>_joints.csv file");
            CorrelationSet CS = make_correlation_set(S);
            correlation_from_files(CS, jf, std::string(jf).replace(at, 6, "prediction"), S.args.count("normalize_time") > 0);
            CS.finalize();
            const std::string out = std::string(jf).replace(at, std::string::npos, "correlations.csv");
            CS.to_csv(out);
            S.log << "Outfile: " << out << "\nDone." << std::endl;
            std::cout << "Done. Log file: " << outfile_log_success << std::endl;
            std::rename(outfile_log.c_str(), outfile_log_success.c_str());
            return EXIT_SUCCESS;
        }
        const std::vector<std::string> param_files = split(S.args["parameter_bounds"], " ");
        std::vector<ParameterSet> params_list;
        for (const auto& pf : param_files) {
            ParameterSet ps(pf, &S.log);
            ps.check_if_complete(S.log);
            S.log << ps << "\n";
            params_list.push_back(ps);
        }
        CsvConfig config(S.args["csv_config"], &S.log);
        S.log << config << "\n";
        S.log << "-> Reading\n";
        LineageTable cells = is_binary_forest(S.args["infile"])
                                 ? read_binary_forest(S.args["infile"], config, S.args["noise_model"], S.args["cell_division_model"], S.log)
                                 : read_data(S.args["infile"], config, S.args["noise_model"], S.args["cell_division_model"], S.log);
        const std::vector<int> segs = segment_indices(cells, S.log);
        if (segs.size() != param_files.size()) {
            S.log << "(main) ERROR: There are " << segs.size() << " segments, but " << param_files.size() << " parameter files!\n";
            throw std::invalid_argument("Invalide argument");
        }
        auto file_number = [&](size_t i) { return segs.size() > 1 ? (int)i : -1; };

        if (S.args.count("minimize"))
            for (size_t i = 0; i < segs.size(); ++i) {
                if (!params_list[i].has_nonfixed()) continue;
                LineageTable slice = get_segment(cells, segs[i]);
                build_genealogy(slice, S.log);
                run_minimization(S, slice, params_list[i], file_number(i));
            }
        if (S.args.count("scan"))
            for (size_t i = 0; i < segs.size(); ++i) {
                LineageTable slice = get_segment(cells, segs[i]);
                build_genealogy(slice, S.log);
                run_bound_1dscan(S, slice, params_list[i], file_number(i));
            }
        if (S.args.count("predict")) {
            build_genealogy(cells, S.log);
            const std::unique_ptr<Forest> F = make_forest(S, cells);
            run_prediction_segments(S, *F, params_list);
            if (S.args.count("joints")) run_joint_distribution(S, *F, params_list);   // needs the predictions on the device
            if (S.args.count("correlation")) run_correlation(S, *F, params_list);
        }
        S.log << "Done." << std::endl;
        std::cout << "Done. Log file: " << outfile_log_success << std::endl;
        std::rename(outfile_log.c_str(), outfile_log_success.c_str());
        S.log.close();
        return EXIT_SUCCESS;
    } catch (std::exception& e) {
        if (!outfile_log.empty()) std::rename(outfile_log.c_str(), outfile_log_error.c_str());
        S.log << "Quit because of an error: " << e.what() << "\n";
        S.log.close();
        std::cout << "Quit because of an error: " << e.what() << "\n";
        std::cout << "Error log file: " << outfile_log_error << std::endl;
        return EXIT_FAILURE;
    }
}
