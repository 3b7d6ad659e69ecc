/* ggp_b200.h — C ABI of libggp_b200.so: the B200 (sm_100a, FP64) implementation of the lineage-tree
 * likelihood / forward-backward / joints hot path of bjks/gfp_gaussian_process.
 *
 * The reference has no plugin or FFI interface; the seam is a set of free C++ functions that walk
 * `std::vector<MOMAdata>` with raw pointers (SURVEY.md §8b).  Each entry point below names the
 * reference function it replaces (paths relative to the reference's src/).  Plain pointers and sizes
 * only; no C++ or torch types; no exceptions cross this boundary (status codes + ggp_last_error()).
 * INTEGRATION.md shows the binding a maintainer would add to the reference's likelihood.h/main.cpp.
 *
 * All host arrays stay owned by the caller and may be freed after the call that takes them returns.
 * Calls on one handle must be serialised by the caller (the reference itself is single-threaded,
 * likelihood.h:7-10).  There is NO CPU fallback: without a CUDA device every call returns
 * GGP_ERR_CUDA.
 */
#ifndef GGP_B200_H
#define GGP_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define GGP_N_PARAMS 11   /* mean_lambda gamma_lambda var_lambda mean_q gamma_q var_q beta var_x var_g var_dx var_dg
                             (likelihood.h:40-42, Parameters.h:175) */

enum {
    GGP_OK = 0,
    GGP_ERR_BAD_ARG = 1,   /* reference: std::invalid_argument */
    GGP_ERR_NAN = 2,       /* reference: std::domain_error("Likelihood is Nan"), likelihood.h:71-93 */
    GGP_ERR_CUDA = 3,
    GGP_ERR_NOMEM = 4
};

enum { GGP_NOISE_CONST = 0, GGP_NOISE_SCALED = 1 };       /* MOMAdata::noise_model, likelihood.h:59-64 */
enum { GGP_DIVISION_GAUSS = 0, GGP_DIVISION_BINOMIAL = 1 }; /* MOMAdata::cell_division_model, predictions.h:40-60 */

/* likelihood arithmetic of a handle (ggp_forest_set_mode).
 * STRICT (default): every result is bit-identical to the reference's own arithmetic (same operation order, glibc's exp /
 *   pow / log bits, no FMA): the path every parity claim is made on; predictions and joints always use it.
 * FAST: ggp_loglik / ggp_loglik_device without root_carry only.  Same model, same moments, evaluated by Gauss-Legendre
 *   quadrature of the integrals of mean_cov_model.h:9-67 and centred covariance formulas, FMA allowed: NOT bit-identical;
 *   it differs from the reference by the reference's own rounding noise (|dloglik| / |loglik| <= 1e-10 is the gate,
 *   DESIGN.md).  A parameter vector whose time steps leave the rule's validity range, or that meets a NaN term, is re-run
 *   on the strict path inside ggp_loglik, so NaN reports are always the reference's.
 * GGP_MODE_FAST picks the smallest rule of {4, 5, 6, 8, 10} nodes that covers the call's parameter vectors on this forest
 * (an a-priori bound; the kernels check every step, and a vector that still leaves the range climbs to the next rule, then to
 * the strict path).  A value N in {4, 5, 6, 8, 10} forces the N-node rule.  ggp_loglik_device, which sees no host
 * parameters, uses the rule the last ggp_loglik chose (6 nodes before any). */
enum { GGP_MODE_STRICT = 0, GGP_MODE_FAST = 1 };

typedef struct ggp_forest ggp_forest;

/* The data the path reads from std::vector<MOMAdata> (moma_input.h:22-80), flattened to SoA.
 * Cells are in input-file order (that order defines daughter1/daughter2 and the depth-first
 * evaluation order, moma_input.h:125-151, likelihood.h:110-122). */
typedef struct {
    int64_t n_cells;
    int64_t n_ctp;               /* total cell-timepoints */
    const int64_t* cell_offset;  /* [n_cells+1] */
    const int32_t* parent;       /* [n_cells] index or -1 */
    const int32_t* daughter1;    /* [n_cells] index or -1 */
    const int32_t* daughter2;    /* [n_cells] index or -1 */
    const double* time;          /* [n_ctp] MOMAdata::time (already divided by rescale_time) */
    const double* log_length;    /* [n_ctp] MOMAdata::log_length */
    const double* fp;            /* [n_ctp] MOMAdata::fp */
    const int32_t* segment;      /* [n_ctp] MOMAdata::segment, or NULL = all 0 */
    int32_t noise_model;
    int32_t division_model;
    double fp_auto;
    /* init_cells_f / init_cells_r statistics (moma_input.h:675-735): mean_x0, mean_g0, var_x0, var_g0 of the
     * first (init_f) and last (init_r) point of all cells with more than one point.  They are population
     * statistics of the WHOLE data set, so a caller that shards trees over processes computes them once
     * globally; set compute_init = 1 to have the library derive them from this forest alone. */
    double init_f[4];
    double init_r[4];
    int32_t compute_init;
    int32_t device;              /* CUDA device ordinal */
} ggp_forest_desc;

/* first point, in the reference's depth-first order, after which the running sum is NaN (likelihood.h:71) */
typedef struct {
    int64_t cell;     /* index into the caller's cell order, -1 if none */
    int64_t t_index;  /* time index inside that cell */
} ggp_nan_info;

/* replaces: read_data -> get_segment -> build_cell_genealogy -> init_cells hand-over (main.cpp:385-411) */
int ggp_forest_create(const ggp_forest_desc* desc, ggp_forest** out);
void ggp_forest_destroy(ggp_forest* f);
/* CUDA stream (cudaStream_t) all work of this handle is enqueued on; NULL = the default stream */
int ggp_forest_set_stream(ggp_forest* f, void* cuda_stream);
int64_t ggp_forest_n_cells(const ggp_forest* f);
int64_t ggp_forest_n_ctp(const ggp_forest* f);
int64_t ggp_forest_n_roots(const ggp_forest* f);
int64_t ggp_forest_n_generations(const ggp_forest* f);
/* replace measurement arrays (MOMAdata::time/log_length/fp, [n_ctp] each, same topology) from host memory; a NULL array
 * is left as it is (an unchanged time grid need not travel again).  The copies are chunked and asynchronous on an internal
 * copy stream when the source is pinned, and the next ggp_loglik starts on a chunk's trees as soon as that chunk has landed
 * (the caller must keep the host arrays alive until that call returns).
 * The root / leaf priors are statistics of the measurements (init_cells_f/r, moma_input.h:675-735), so new log_length / fp
 * arrays come with new statistics: pass them (init_f4, init_r4, e.g. from ggp_init_stats over the whole data set), or pass
 * NULL, NULL to have the library re-derive them from the new arrays - possible only for a forest created with
 * compute_init = 1 (one host pass over the cells' first and last points); a forest created with the statistics of a larger
 * data set (compute_init = 0) returns GGP_ERR_BAD_ARG instead of silently keeping stale priors.
 * Used when the same genealogy is evaluated on new measurements (and by bench.py's end-to-end leg). */
int ggp_forest_upload_series(ggp_forest* f, const double* time, const double* log_length, const double* fp,
                             const double* init_f4, const double* init_r4);
int ggp_forest_get_init(const ggp_forest* f, double* init_f4, double* init_r4);
/* likelihood arithmetic of this handle: GGP_MODE_STRICT (default), GGP_MODE_FAST, or a node count (see above); also set by
 * the environment variable GGP_B200_FAST at ggp_forest_create */
int ggp_forest_set_mode(ggp_forest* f, int32_t mode);
int32_t ggp_forest_get_mode(const ggp_forest* f);   /* the value set: 0 strict, 1 fast, or a forced node count */
int32_t ggp_last_fast_nodes(const ggp_forest* f);   /* node count GGP_MODE_FAST chose last (or the last ggp_loglik_grad used) */
/* number of parameter vectors of the last fast ggp_loglik that were re-run on the strict path */
int64_t ggp_last_strict_reruns(const ggp_forest* f);
/* the init_cells_f / init_cells_r statistics of a data set (moma_input.h:675-735) without creating a forest: what a caller
 * that shards trees over several handles passes to every shard (compute_init = 0).  Host arithmetic on the descriptor's
 * arrays (input preparation, not part of the device path). */
int ggp_init_stats(const ggp_forest_desc* desc, double* init_f4, double* init_r4);

/* replaces: total_likelihood(params_vec, cells) (likelihood.h:170-174; objective :125-159) for n_vec
 * parameter vectors at once (scan main.cpp:105-108, Hessian stencil likelihood.h:211-258, simplex).
 *   params       [n_vec][11], natural space (the caller applies exp() for log-space search, likelihood.h:161-167)
 *   root_carry   NULL = every vector is a first ("fresh") evaluation; else in/out [n_roots][16] = the roots'
 *                persistent MOMAdata::cov (row-major 4x4): vectors are evaluated as if sequentially, each
 *                root starting from the off-diagonals the previous evaluation left (predictions.h:64-78,
 *                SURVEY.md H3).  Roots are numbered in cell order.
 *   out_loglik   [n_vec] +log-likelihood
 *   out_cell_ll  NULL or [n_vec][n_cells]: each cell's own sum (diagnostics / parity tests)
 *   nan          NULL or [n_vec]
 * returns GGP_ERR_NAN if any vector hit a NaN (all vectors are still evaluated). */
int ggp_loglik(ggp_forest* f, const double* params, int32_t n_vec, double* root_carry,
               double* out_loglik, double* out_cell_ll, ggp_nan_info* nan);

/* same, but params and out_loglik are DEVICE pointers and nothing is copied or synchronised:
 * the evaluation is enqueued on the handle's stream (for callers that keep data resident). */
int ggp_loglik_device(ggp_forest* f, const double* d_params, int32_t n_vec, double* d_out_loglik);

/* gradient of the log-likelihood: d(+log-likelihood) / d(params) at n_vec parameter vectors, natural space, FAST arithmetic
 * whatever the handle's mode (forward-mode dual numbers through the fast step; the strict path's rounding has no meaningful
 * derivative).  No reference counterpart: it serves error bars (a Hessian as central differences of the gradient, 2 n
 * gradients, instead of second differences of the likelihood) and gradient-based fitting.
 *   dirs        NULL = all 11 parameters (n_dirs must be 11), else the n_dirs distinct parameter indices (0 .. 10) to
 *               differentiate, e.g. the free ones
 *   out_loglik  [n_vec] the fast log-likelihood
 *   out_grad    [n_vec][n_dirs], column j = d / d params[dirs[j]]
 *   nan         NULL or [n_vec]
 * The rule: the node count forced on the handle (ggp_forest_set_mode(f, N)), else the smallest that covers the batch
 * (ggp_last_fast_nodes reports it).  A vector that leaves the rule's validity range is evaluated again with the next larger
 * rule.  A vector no rule covers gets the strict log-likelihood and a NaN gradient row, and the call returns GGP_ERR_BAD_ARG
 * (naming the vector in ggp_last_error) after filling every other row; a vector that meets a NaN term gets the strict path's
 * NaN record and a NaN row, and the call returns GGP_ERR_NAN (GGP_ERR_BAD_ARG if both kinds occur).  One thread carries one
 * direction: the cost is about that of 2 n_dirs fast evaluations.  Shares the handle's workspaces; what the other calls
 * return is unaffected. */
int ggp_loglik_grad(ggp_forest* f, const double* params, int32_t n_vec, const int32_t* dirs, int32_t n_dirs,
                    double* out_loglik, double* out_grad, ggp_nan_info* nan);

/* exact Hessian of the fast log-likelihood: value, gradient and second derivatives at n_vec parameter vectors, natural space,
 * FAST arithmetic whatever the handle's mode.  No step size: second-order Taylor numbers (value, first and second derivative
 * along one direction u) run through the fast step, and the mixed derivatives come by polarization from the n (n + 1) / 2
 * directions u = s_i e_i (i in dirs) and s_i e_i + s_j e_j (i < j), with s_i the power of two nearest |params[i]| (1 for 0),
 * so the result is exact up to rounding and symmetric bit for bit (DESIGN.md 5.7).  It serves exact error bars:
 * -diag(inverse(H)) (the command line's --exact_errors).
 *   dirs, n_dirs, out_loglik, nan   as ggp_loglik_grad
 *   out_grad    [n_vec][n_dirs]           column j = d / d params[dirs[j]]
 *   out_hess    [n_vec][n_dirs][n_dirs]   entry (j, k) = d^2 / d params[dirs[j]] d params[dirs[k]]
 * The rule, the re-run ladder, the counters and the error rows are those of ggp_loglik_grad (a vector no rule covers or that
 * meets a NaN term gets NaN gradient and Hessian rows).  A vector's evaluations that do not fit GGP_B200_STATE_BUDGET run in
 * ranges; every evaluation is independent, so a direction subset and every chunking give the same bits.
 * Cost: one evaluation per direction pair (n (n + 1) / 2), each about 5.4 fast evaluations or 2.4 gradient directions; all 11
 * parameters on the configs[1] forest (630 000 cells, resident): 205 ms on one B200 at 1000 W (DESIGN.md 5.7). */
int ggp_loglik_hess(ggp_forest* f, const double* params, int32_t n_vec, const int32_t* dirs, int32_t n_dirs,
                    double* out_loglik, double* out_grad, double* out_hess, ggp_nan_info* nan);

/* replaces: prediction_forward / prediction_backward / combine_predictions (predictions.h:166, 438, 466;
 * main.cpp:132-140).  params [n_seg][11] indexed by MOMAdata::segment.  Each output is NULL or
 * [n_ctp][20] = 4 means + the 4x4 covariance row-major, per ctp in the caller's order; the
 * 14 numbers the reference's writer prints are the mean and the upper triangle (predictions.h:541-552).
 * Device copies are kept in the handle for ggp_joints. */
int ggp_predict(ggp_forest* f, const double* params, int32_t n_seg,
                double* out_forward, double* out_backward, double* out_combined);

/* the same passes with the outputs in the layout the reference's writer prints (predictions.h:575-578): [n_ctp][14] = 4 means +
 * the upper triangle row-major (xx xg xl xq gg gl gq ll lq qq), packed on the device: 30 % fewer bytes to the host */
int ggp_predict14(ggp_forest* f, const double* params, int32_t n_seg,
                  double* out_forward14, double* out_backward14, double* out_combined14);

/* replaces: collect_joint_distributions (correlation_tree.h:629-648) with a sparse result: record r =
 * (row_ctp[r], col_ctp[r], rec[r][44]): the joint P(z_col, z_row | D) as 8 means (z_col then z_row) and the 36
 * upper-triangular covariances row-major, sorted by (row, col) = the order the reference writes its dense CSV in.
 * Rows are the start points row_begin <= ctp < row_end, so a caller can stream the matrix in row blocks like the
 * reference streams lines (the dense row of the example data set alone is 22 065 x 44 fields).  Requires a prior
 * ggp_predict on the handle with the same params.  *out_count receives the number of joints the rows hold; at most
 * `cap` are written (call with cap = 0 to size the buffers).  The call's device scratch (about 800 bytes per record) stays with
 * the handle for the next call as long as it is below 6 GB, and goes with ggp_forest_destroy. */
int ggp_joints(ggp_forest* f, const double* params, int32_t n_seg, double rel_tol, int64_t row_begin, int64_t row_end,
               int64_t cap, int64_t* out_count, int64_t* row_ctp, int64_t* col_ctp, double* rec44);

/* replaces: the accumulation of python_src/correlation_from_joint.py (Correlation.add_gaussian :287-302, files2correlation_function
 * :443-560 with the product-of-marginals fallback :528-534) on top of collect_joint_distributions: the lag-binned moment sums of
 * the correlation functions straight from the walk, without a joints file or a record ever leaving the device.
 * Lag bins k * dt_step, k = 0 .. n_bins - 1 (np.arange(0, dt * n_data, dt)); a pair (row i, column j on i's lineage, j > i, or any
 * emitted joint) goes to the first bin with |k dt_step - dt| <= atol + 1e-5 |dt| (np.isclose; the script uses atol = 0.2 dt_step),
 * dt = time[j] - time[i], divided by the row cell's life time if normalize_time; lag 0 takes every point with itself.
 *   out_sums [n_bins][50] = n, sum m[8], sum (m m^T + C) upper triangle row-major [36], sum c[2], sum c c^T upper [3] with
 *                           c = g / exp(x), indices 0..3 = z(t + dt), 4..7 = z(t); accumulated with compensation on the device,
 *                           per-block partials added in long double; each entry is the leading double of its sum,
 *   out_sums_lo             NULL or [n_bins][50]: the remainder (sum - leading double),
 *   out_joints              NULL or the number of joints the walk emitted.
 * The joints are walked in row blocks whose records stay on the device; their buffers (a quarter of the free device memory,
 * at most 16 GB, by default) stay with the handle until ggp_forest_destroy.
 * Requires a prior ggp_predict with the same params, fewer than 65 535 bins, and parents stored before their daughters (else
 * GGP_ERR_BAD_ARG: reduce the sparse records of ggp_joints on the host, host/ggp_correlation.hpp). */
int ggp_correlation_sums(ggp_forest* f, const double* params, int32_t n_seg, double rel_tol, double dt_step, int32_t n_bins,
                         double atol, int32_t normalize_time, double* out_sums, double* out_sums_lo, int64_t* out_joints);

/* ---- one host process, several GPUs (SURVEY.md 8b "Threading", 8e) ---------------------------------------------------------
 * A group shards the lineage trees of ONE data set over devices behind one handle: every shard is a ggp_forest on its own
 * device (own streams, one host thread per shard inside a call), created with the init_cells statistics of the whole data set;
 * the per-shard log-likelihoods are added on the host in shard order (reproducible; 8 bytes per vector need no collective),
 * per-cell sums, root_carry and prediction rows come back in the caller's order.  A data set stored tree by tree is split into
 * contiguous runs of trees, so each device copies its prediction rows straight into their place in the caller's arrays;
 * otherwise trees are bin-packed by size and the rows are scattered back by index.  Same argument meaning and error
 * behaviour as the single-forest calls (ggp_group_member + ggp_group_member_ctp give the members' handles and
 * index maps).  `devices` may name a device more than once. */
typedef struct ggp_group ggp_group;
int ggp_group_create(const ggp_forest_desc* desc, const int32_t* devices, int32_t n_devices, ggp_group** out);   /* desc->device is ignored */
void ggp_group_destroy(ggp_group* g);
int32_t ggp_group_size(const ggp_group* g);
int32_t ggp_group_is_contiguous(const ggp_group* g);
ggp_forest* ggp_group_member(ggp_group* g, int32_t k);                             /* NULL: shard k holds no tree */
int64_t ggp_group_member_cells(const ggp_group* g, int32_t k, int64_t* cells);     /* caller's cell index of the shard's cells; NULL: count only */
int64_t ggp_group_member_ctp(const ggp_group* g, int32_t k, int64_t* ctp);         /* caller's time-point index of the shard's time points */
int ggp_group_set_mode(ggp_group* g, int32_t mode);
int ggp_group_loglik(ggp_group* g, const double* params, int32_t n_vec, double* root_carry, double* out_loglik,
                     double* out_cell_ll, ggp_nan_info* nan);
/* ggp_loglik_grad over the shards: values and gradients added on the host in shard order */
int ggp_group_loglik_grad(ggp_group* g, const double* params, int32_t n_vec, const int32_t* dirs, int32_t n_dirs,
                          double* out_loglik, double* out_grad, ggp_nan_info* nan);
/* ggp_loglik_hess over the shards: values, gradients and Hessians added on the host in shard order */
int ggp_group_loglik_hess(ggp_group* g, const double* params, int32_t n_vec, const int32_t* dirs, int32_t n_dirs,
                          double* out_loglik, double* out_grad, double* out_hess, ggp_nan_info* nan);
int ggp_group_predict(ggp_group* g, const double* params, int32_t n_seg, double* out_forward, double* out_backward, double* out_combined);
int ggp_group_predict14(ggp_group* g, const double* params, int32_t n_seg, double* out_forward14, double* out_backward14,
                        double* out_combined14);
/* ggp_joints over the shards (collect_joint_distributions, correlation_tree.h:629-648): rows, columns and the row range are the
 * CALLER's time-point indices, records sorted by (row, col); requires a prior ggp_group_predict[14] with the same params.  Every
 * shard counts first: if the total exceeds `cap` only *out_count is written. */
int ggp_group_joints(ggp_group* g, const double* params, int32_t n_seg, double rel_tol, int64_t row_begin, int64_t row_end, int64_t cap,
                     int64_t* out_count, int64_t* row_ctp, int64_t* col_ctp, double* rec44);
/* ggp_correlation_sums over the shards: the sums run over pairs of points of one lineage tree, so they add over shards */
int ggp_group_correlation_sums(ggp_group* g, const double* params, int32_t n_seg, double rel_tol, double dt_step, int32_t n_bins,
                               double atol, int32_t normalize_time, double* out_sums, double* out_sums_lo, int64_t* out_joints);

/* waits for the evaluation enqueued by ggp_loglik_device and returns its device time in milliseconds */
int ggp_sync_kernel_ms(ggp_forest* f, double* ms_out);

/* each cell's MOMAdata::mean/cov as prediction_backward leaves them ([n_cells][20], caller's cell order, 4 means +
 * 4x4 row-major, in the backward pass's sign-flipped frame); collect_joint_distributions reads them
 * (correlation_tree.h:519-524, SURVEY.md H3).  Requires a prior ggp_predict. */
int ggp_backward_cell_state(ggp_forest* f, double* out_cell_state20);

/* last device kernel time of the handle in milliseconds (CUDA events around the launches of the last call) */
double ggp_last_kernel_ms(const ggp_forest* f);
/* number of kernel launches issued by the last call */
int64_t ggp_last_launch_count(const ggp_forest* f);

const char* ggp_last_error(void);
const char* ggp_version(void);

/* device self-test of the strict math (exp/log/pow/Dawson/propagate) for callers that hold expected bits:
 * evaluates fn over n inputs on the device.  fn: 0 exp, 1 log, 2 pow(x, y), 3 dawson, 4 x / y through the shared-reciprocal
 * divisor path (GgpDivisor).  y may be NULL for 0, 1, 3, 6.
 * 5: the interleaved pow + exp block of the cooperative step: out[5 i] = pow(x[i], 1.5 + i % 3), out[5 i + 1..4] = exp of
 *    y[i], y[i] / 2, -y[i], y[i] + 1 (out holds 5 n doubles).
 * 6: the log-evidence term (likelihood.h:26-32) as the cooperative step finishes it inside a phase: x holds 5 n doubles
 *    (quadratic form -1/2 r^T S^-1 r, S00, S01, S10, S11 per case), out[i] = the term. */
int ggp_math_eval(int32_t device, int32_t fn, int64_t n, const double* x, const double* y, double* out);
/* propagate n independent states (14 doubles each: 4 means + upper triangle) over dt[i] with 7 OU params each
 * (mean_cov_model, mean_cov_model.h:211); cross (NULL or [n][16]) receives cross_cov_model (:380). */
int ggp_propagate_eval(int32_t device, int64_t n, const double* state14, const double* dt, const double* p7,
                       double* out14, double* cross16);

/* measured FP64 FMA throughput of the device in TFLOP/s (register-resident DFMA chains, best of 5): the
 * roofline denominator of this path, which is bound by the FP64 pipe (SURVEY.md 8d) */
int ggp_fp64_peak(int32_t device, double* tflops_out);

#ifdef __cplusplus
}
#endif
#endif
