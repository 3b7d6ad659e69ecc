// ggp_b200.cu — C ABI of libggp_b200.so (include/ggp_b200.h): host-side flattening of the lineage forest
// into generation-ordered device arrays, launch sequencing, and result hand-back.
//
// Host side of what the reference does in moma_input.h:125-189 (genealogy, roots), likelihood.h:110-174
// (depth-first evaluation order; here only used to report the first NaN and to order nothing else) and
// main.cpp:115-145 (forward, backward, combine).  No CPU compute path exists in this library: every
// numerical result comes from the library's kernels (ggp_coop_kernels.cuh and ggp_fast.cu for the likelihood and the
// prediction passes, ggp_kernels.cuh, ggp_joints.cuh).
//
// Build: nvcc -std=c++17 -O3 -fmad=false -gencode arch=compute_100a,code=sm_100a -lineinfo -shared
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iterator>
#include <numeric>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/ggp_b200.h"
#include "ggp_layout.hpp"
#include "ggp_kernels.cuh"
#include "ggp_coop_kernels.cuh"
#include "ggp_joints.cuh"
#include "ggp_fast_api.h"

// groups per block of the prediction passes: 3 (384 threads, up to 170 registers) keeps their larger per-thread state
// (segment lookups, output pointers) out of local memory; with 4 groups the 128-register cap spills loop-carried values
// and, with the L1 carve-out almost entirely shared memory, every reload goes to L2
constexpr int kPredNG = 3;
constexpr int kPredUniNG = 4;   // groups per block of the one-segment prediction kernels (uniform parameters)

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

#define GGP_CUDA(call)                                                                             \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(e_ == cudaErrorMemoryAllocation ? GGP_ERR_NOMEM : GGP_ERR_CUDA,            \
                        std::string(#call) + ": " + cudaGetErrorString(e_));                       \
    } while (0)

template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }   // scratch buffers of a call are freed on every return path
    cudaError_t ensure(size_t count) {
        if (count <= n) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
        cudaError_t e = cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T));
        if (e == cudaSuccess) n = count;
        return e;
    }
    cudaError_t upload(const std::vector<T>& h, cudaStream_t s) {
        cudaError_t e = ensure(h.size());
        if (e != cudaSuccess) return e;
        return cudaMemcpyAsync(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, s);
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
    }
};

struct ScopedEvent {
    cudaEvent_t ev = nullptr;
    ScopedEvent() = default;
    ScopedEvent(const ScopedEvent&) = delete;
    ScopedEvent& operator=(const ScopedEvent&) = delete;
    ~ScopedEvent() { if (ev) cudaEventDestroy(ev); }
    cudaError_t create() { return cudaEventCreate(&ev); }
};

}  // namespace

struct ggp_forest {
    int device = 0;
    cudaStream_t stream = nullptr;
    int64_t n_cells = 0, n_ctp = 0;
    int32_t n_roots = 0, n_gen = 0, max_seg = 0;
    GgpModel model{};
    GgpLayout L;                          // host topology
    std::vector<int32_t> gen_partial0;    // [n_gen][n_chunks+1] first block partial of each (generation, upload chunk); 32 cells per partial
    int32_t n_partial = 0;
    // streamed upload (ggp_forest_upload_series): chunked copies on their own stream, one event per chunk
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t pass_done[3] = {nullptr, nullptr, nullptr};   // ggp_predict: forward / backward / combined output complete
    std::vector<cudaEvent_t> chunk_ready;
    cudaEvent_t compute_done = nullptr;
    // streamed evaluation: chunk k's launches run on chunk_stream[k] (the last chunk on the handle's stream), so that the
    // small early generations of one chunk (a few blocks, latency bound) run beside the large late generations of another
    std::vector<cudaStream_t> chunk_stream;
    std::vector<cudaEvent_t> chunk_done;
    cudaEvent_t eval_start = nullptr;
    bool upload_pending = false;
    bool compute_init = false;            // created with compute_init = 1: upload_series re-derives the init_cells statistics
    std::vector<double> edge;             // [4][n_cells] first x, last x, first g, last g of every cell (host copy for that re-derivation)
    std::vector<int64_t> h_off;           // [n_cells+1] caller's cell offsets (kept with `edge`)
    int64_t coop_ng4_min_groups = 0;      // launches with at least this many 32-cell groups use 4 groups per block (8 per SM; set at create)
    int fast_mode = 0;                    // ggp_forest_set_mode / GGP_B200_FAST: 0 strict (bit-exact, the default), 1 fast with the node
                                          // count chosen per call from the parameters and the forest's largest time step, N = fast with an
                                          // N-node rule; not bit-exact, fresh-mode ggp_loglik only
    int auto_nodes = GGP_FAST_DEFAULT_NODES;   // what mode 1 chose last (ggp_loglik_device, which sees no host parameters, uses it)
    int last_nodes = GGP_FAST_DEFAULT_NODES;   // ggp_last_fast_nodes: auto_nodes after ggp_loglik, the rule ggp_loglik_grad / _hess started with after it
    double dt_max = 0.0;                  // largest time step of the forest
    // the forest's distinct time steps and, per time point, the index of the step that arrives there (fast likelihood)
    std::vector<double> dt_values;
    bool dt_ok = false;                   // false: more than 65 534 distinct steps, the fast mode is unavailable (strict is used)
    DevBuf<uint16_t> dt_idx;
    DevBuf<double> d_dt_values;
    DevBuf<unsigned char> w_ktab;
    int32_t device_fast_vecs = 0;         // vectors of a fast ggp_loglik_device whose flags ggp_sync_kernel_ms still has to read
    // device
    DevBuf<double> time, x, g;
    DevBuf<int32_t> seg, comb_seg;
    DevBuf<int64_t> s_off, s_dfs0;
    DevBuf<int32_t> s_n, s_parent, s_d1, s_d2, s_root, s_cell;
    // workspaces
    DevBuf<double> w_params, w_state, w_partial, w_out, w_cell_ll, w_carry;
    DevBuf<unsigned long long> w_nan;
    DevBuf<int> w_invalid;
    DevBuf<double> fwd, bwd, comb, bstate, pred_params, prep, jstack, pack;
    DevBuf<int32_t> ctp_slot, jstack_slot;
    // scratch of ggp_correlation_sums, kept between calls (a row block's records alone are 1.5 GB: allocating and freeing
    // them per call cost more than the kernels)
    struct {
        DevBuf<long long> row, col;
        DevBuf<double> rec, partial;
        DevBuf<unsigned long long> count;
        DevBuf<unsigned short> key, key2;
        DevBuf<unsigned int> idx, idx2;
        DevBuf<unsigned char> tmp;
    } corr;
    // scratch of ggp_joints, kept between calls while it stays below GGP_JOINT_SCRATCH_KEEP bytes (the command line fetches row
    // block after row block: allocating and freeing ~2 GB per call cost more than the walk; a single huge call gives it back)
    struct {
        DevBuf<long long> row, col, row2, col2;
        DevBuf<double> rec, rec2;
        DevBuf<unsigned long long> count, key, key2;
        DevBuf<unsigned int> idx, idx2;
        DevBuf<unsigned char> tmp;
        size_t bytes() const {
            return (row.n + col.n + row2.n + col2.n + rec.n + rec2.n + count.n + key.n + key2.n) * 8 + (idx.n + idx2.n) * 4 + tmp.n;
        }
        void release() {
            row.release(); col.release(); row2.release(); col2.release(); rec.release(); rec2.release(); count.release();
            key.release(); key2.release(); idx.release(); idx2.release(); tmp.release();
        }
    } jscratch;
    bool have_prep = false;
    bool have_pred = false;
    int32_t pred_n_seg = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // counters of the last call.  last_ms: its device time; for ggp_loglik, ggp_loglik_grad and ggp_loglik_hess the sum over their passes (ev0 ->
    // ev1 of each).  last_launches: its kernel launches; for an evaluation the sum of its passes' enqueue_loglik launches (the
    // fills of keys, flags and partials are not counted).  last_reruns: the vectors of a fast ggp_loglik or of ggp_loglik_grad / _hess
    // that the strict kernels evaluated.
    double last_ms = 0.0;
    int64_t last_launches = 0;
    int64_t last_reruns = 0;
    int64_t state_budget_bytes = (int64_t)8 << 30;   // end-of-cell state of one vector chunk (n_vec * n_cells * 112 B); GGP_B200_STATE_BUDGET overrides (bytes)
    int n_sm = 0;                 // cudaDevAttrMultiProcessorCount of the handle's device
    int walk_blocks_per_sm = 1;   // joints walker blocks (256 threads) resident per SM (register-limited); GGP_B200_WALK_BLOCKS overrides
    int64_t walk_total_blocks = 0;   // GGP_B200_WALK_TOTAL_BLOCKS: cap on the number of walker blocks (tests: results do not depend on it)
    unsigned fill_grid(size_t cnt) const { return (unsigned)std::max<size_t>(1, std::min<size_t>((cnt + 255) / 256, (size_t)n_sm * 8)); }

    GgpDevForest dev() const {
        GgpDevForest F;
        F.n_cells = n_cells; F.n_ctp = n_ctp;
        F.time = time.p; F.x = x.p; F.g = g.p; F.seg = seg.p;
        F.s_off = s_off.p; F.s_n = s_n.p; F.s_parent = s_parent.p; F.s_d1 = s_d1.p; F.s_d2 = s_d2.p;
        F.s_root = s_root.p; F.s_cell = s_cell.p; F.s_dfs0 = s_dfs0.p;
        F.model = model;
        for (int i = 0; i < 4; ++i) { F.init_f[i] = L.init_f[i]; F.init_r[i] = L.init_r[i]; }
        F.dt_idx = dt_idx.p;
        F.n_dt = (int32_t)dt_values.size();
        return F;
    }
};

namespace {

int check_handle(const ggp_forest* f) {
    if (!f) return fail(GGP_ERR_BAD_ARG, "null forest handle");
    return GGP_OK;
}

// table of the distinct time steps of the forest (exact comparison of doubles) and its index per time point; the step that
// arrives at a cell's first point starts at the mother's last point (predictions.h:28-31)
cudaError_t build_dt_table(ggp_forest* f, const double* time) {
    const GgpLayout& L = f->L;
    std::vector<uint16_t> idx((size_t)L.n_ctp, (uint16_t)0xffff);
    std::unordered_map<uint64_t, int> seen;
    f->dt_values.clear();
    f->dt_ok = true;
    uint64_t last_bits = ~0ull;
    int last_i = -1;
    for (int64_t s = 0; s < L.n_cells && f->dt_ok; ++s) {
        const int64_t off = L.s_off[s];
        const int32_t par = L.s_parent[s];
        for (int64_t t = 0; t < L.s_n[s]; ++t) {
            const int64_t from = t > 0 ? off + t - 1 : (par >= 0 ? L.s_off[par] + L.s_n[par] - 1 : -1);
            if (from < 0) continue;
            const double dt = time[off + t] - time[from];
            uint64_t bits;
            std::memcpy(&bits, &dt, 8);
            if (bits != last_bits) {
                auto it = seen.find(bits);
                if (it == seen.end()) {
                    if (f->dt_values.size() >= 65534) { f->dt_ok = false; break; }
                    it = seen.emplace(bits, (int)f->dt_values.size()).first;
                    f->dt_values.push_back(dt);
                }
                last_bits = bits;
                last_i = it->second;
            }
            idx[(size_t)(off + t)] = (uint16_t)last_i;
        }
    }
    if (!f->dt_ok) { f->dt_values.clear(); return cudaSuccess; }
    f->dt_max = 0.0;
    for (double v : f->dt_values) f->dt_max = std::max(f->dt_max, std::fabs(v));
    cudaError_t e = f->dt_idx.ensure(idx.size());
    if (e == cudaSuccess) e = cudaMemcpy(f->dt_idx.p, idx.data(), idx.size() * sizeof(uint16_t), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = f->d_dt_values.ensure(std::max<size_t>(f->dt_values.size(), 1));
    if (e == cudaSuccess && !f->dt_values.empty())
        e = cudaMemcpy(f->d_dt_values.p, f->dt_values.data(), f->dt_values.size() * sizeof(double), cudaMemcpyHostToDevice);
    return e;
}

int grid_of(int64_t n) { return (int)((n + GGP_BLOCK - 1) / GGP_BLOCK); }
int grid_of_coop(int64_t n) { return (int)((n + GGP_COOP_CELLS - 1) / GGP_COOP_CELLS); }

// the pass kernels use ~100 kB of dynamic shared memory per block (tables + per-thread scratch): opt in once per device
cudaError_t opt_in_smem() {
    cudaError_t e = cudaFuncSetAttribute(ggp_loglik_coop_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GGP_COOP_SMEM_BYTES(1));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ggp_loglik_coop_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GGP_COOP_SMEM_BYTES(4));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ggp_loglik_coop_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GGP_COOP_SMEM_BYTES(1));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ggp_loglik_coop_kernel<kPredNG, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GGP_COOP_SMEM_BYTES(kPredNG));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ggp_loglik_coop_kernel<kPredUniNG, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GGP_COOP_SMEM_BYTES(kPredUniNG));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ggp_backward_coop_kernel<kPredUniNG, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GGP_COOP_SMEM_BYTES(kPredUniNG));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ggp_backward_coop_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GGP_COOP_SMEM_BYTES(1));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ggp_backward_coop_kernel<kPredNG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GGP_COOP_SMEM_BYTES(kPredNG));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ggp_loglik_chain_coop_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GGP_COOP_SMEM_BYTES_CHAIN);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ggp_coop_math_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GGP_COOP_SMEM_BYTES(1));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ggp_joint_prep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GGP_SMEM_BYTES);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ggp_propagate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GGP_SMEM_BYTES);
    return e;
}

}  // namespace

extern "C" {

const char* ggp_last_error(void) { return g_err.c_str(); }
const char* ggp_version(void) { return "ggp-b200 0.1 (sm_100a, fp64 strict)"; }

int ggp_forest_create(const ggp_forest_desc* d, ggp_forest** out) {
    if (!d || !out) return fail(GGP_ERR_BAD_ARG, "null argument");
    *out = nullptr;
    ggp_forest* f = new ggp_forest();
    // measured on cfg2, end to end per step: one stream for all chunks 1 -> 11.6 ms, 2 -> 9.7, 3 -> 9.0 (8.47 with the final
    // kernels), 4 -> 9.7, 8 -> 11.7; one stream per chunk (chunk_stream): 3 -> 8.25, 6 -> 7.95, 8 / 12 -> 7.93; the copy
    // alone takes 5.5 ms (55 GB/s), the evaluation keeps up with it at ~80 % of its resident rate (per-chunk event timeline:
    // every chunk's launches take ~2.2 ms, three chunks in flight), small first chunks do not help
    int32_t want_chunks = d->n_ctp >= (int64_t)2000000 ? 6 : 1;
    if (const char* m = getenv("GGP_B200_UPLOAD_CHUNKS")) want_chunks = atoi(m);
    std::vector<double> fractions;   // GGP_B200_CHUNK_FRACTIONS=a,b,c,...: relative chunk sizes (A/B measurements)
    if (const char* m = getenv("GGP_B200_CHUNK_FRACTIONS")) {
        for (const char* q = m; *q;) {
            char* end = nullptr;
            const double v = strtod(q, &end);
            if (end == q) break;
            if (v > 0.0) fractions.push_back(v);
            q = (*end == ',') ? end + 1 : end;
        }
        if (!fractions.empty()) want_chunks = (int32_t)fractions.size();
    }
    const std::string why = f->L.build(d, want_chunks, fractions.empty() ? nullptr : fractions.data());
    if (!why.empty()) {
        delete f;
        return fail(GGP_ERR_BAD_ARG, why);
    }
    int dev_count = 0;
    cudaError_t e = cudaGetDeviceCount(&dev_count);
    if (e != cudaSuccess || d->device < 0 || d->device >= dev_count) {
        delete f;
        return fail(GGP_ERR_CUDA, e != cudaSuccess ? std::string("no CUDA device: ") + cudaGetErrorString(e) : "no such CUDA device");
    }
    e = cudaSetDevice(d->device);
    if (e == cudaSuccess) e = opt_in_smem();
    const GgpLayout& L = f->L;
    f->device = d->device;
    f->n_cells = L.n_cells;
    f->n_ctp = L.n_ctp;
    f->n_roots = L.n_roots;
    f->n_gen = L.n_gen;
    f->max_seg = L.max_seg;
    f->model.noise_scaled = d->noise_model == GGP_NOISE_SCALED;
    f->model.division_binomial = d->division_model == GGP_DIVISION_BINOMIAL;
    f->model.fp_auto = d->fp_auto;
    f->compute_init = d->compute_init != 0;
    if (f->compute_init) {
        f->edge.resize((size_t)4 * L.n_cells);
        f->h_off.assign(d->cell_offset, d->cell_offset + L.n_cells + 1);
        for (int64_t c = 0; c < L.n_cells; ++c) {
            const int64_t o = d->cell_offset[c], l = d->cell_offset[c + 1] - 1;
            f->edge[c] = d->log_length[o];
            f->edge[L.n_cells + c] = d->log_length[l];
            f->edge[2 * L.n_cells + c] = d->fp[o];
            f->edge[3 * L.n_cells + c] = d->fp[l];
        }
    }
    {
        const int K = L.n_chunks;
        f->gen_partial0.assign((size_t)L.n_gen * (K + 1), 0);
        int32_t acc = 0;
        for (int g = 0; g < L.n_gen; ++g)
            for (int k = 0; k <= K; ++k) {
                f->gen_partial0[(size_t)g * (K + 1) + k] = acc;
                if (k < K) acc += grid_of_coop(L.gen_chunk_start[(size_t)g * (K + 1) + k + 1] - L.gen_chunk_start[(size_t)g * (K + 1) + k]);
            }
        f->n_partial = acc;
    }
    {
        int n_sm = 0;
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, f->device);
        f->n_sm = std::max(n_sm, 1);
        f->coop_ng4_min_groups = (int64_t)4 * f->n_sm * 2;
        if (const char* m = getenv("GGP_B200_NG4_MIN")) f->coop_ng4_min_groups = atoll(m);
        if (const char* m = getenv("GGP_B200_WALK_BLOCKS")) f->walk_blocks_per_sm = std::max(1, atoi(m));
        if (const char* m = getenv("GGP_B200_WALK_TOTAL_BLOCKS")) f->walk_total_blocks = std::max<int64_t>(0, atoll(m));
        if (const char* m = getenv("GGP_B200_STATE_BUDGET")) f->state_budget_bytes = std::max<int64_t>(1, atoll(m));
        if (const char* m = getenv("GGP_B200_FAST")) {   // 1 = the default rule, N = an N-node rule
            const int n = atoi(m);
            f->fast_mode = n == 1 ? 1 : (ggp_fast_supported_nodes(n) ? n : 0);
        }
    }

    cudaStream_t s = nullptr;
    auto up_d = [&](DevBuf<double>& b, const double* h, int64_t n) {
        if (e != cudaSuccess) return;
        e = b.ensure(n);
        if (e == cudaSuccess) e = cudaMemcpyAsync(b.p, h, n * sizeof(double), cudaMemcpyHostToDevice, s);
    };
    up_d(f->time, d->time, d->n_ctp);
    up_d(f->x, d->log_length, d->n_ctp);
    up_d(f->g, d->fp, d->n_ctp);
    if (e == cudaSuccess) e = f->seg.upload(L.seg, s);
    if (e == cudaSuccess) e = f->comb_seg.upload(L.comb_seg, s);
    if (e == cudaSuccess) e = f->s_off.upload(L.s_off, s);
    if (e == cudaSuccess) e = f->s_dfs0.upload(L.s_dfs0, s);
    if (e == cudaSuccess) e = f->s_n.upload(L.s_n, s);
    if (e == cudaSuccess) e = f->s_parent.upload(L.s_parent, s);
    if (e == cudaSuccess) e = f->s_d1.upload(L.s_d1, s);
    if (e == cudaSuccess) e = f->s_d2.upload(L.s_d2, s);
    if (e == cudaSuccess) e = f->s_root.upload(L.s_root, s);
    if (e == cudaSuccess) e = f->s_cell.upload(L.s_cell, s);
    if (e == cudaSuccess) e = f->ctp_slot.upload(L.ctp_slot, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e == cudaSuccess) e = build_dt_table(f, d->time);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&f->copy_stream, cudaStreamNonBlocking);
    for (int o = 0; o < 3 && e == cudaSuccess; ++o) e = cudaEventCreateWithFlags(&f->pass_done[o], cudaEventDisableTiming);
    f->chunk_ready.assign(L.n_chunks, nullptr);
    for (int k = 0; k < L.n_chunks && e == cudaSuccess; ++k) e = cudaEventCreateWithFlags(&f->chunk_ready[k], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&f->compute_done, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&f->eval_start, cudaEventDisableTiming);
    if (L.n_chunks > 1) {
        f->chunk_stream.assign(L.n_chunks - 1, nullptr);
        f->chunk_done.assign(L.n_chunks - 1, nullptr);
        for (int k = 0; k + 1 < L.n_chunks && e == cudaSuccess; ++k) {
            e = cudaStreamCreateWithFlags(&f->chunk_stream[k], cudaStreamNonBlocking);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&f->chunk_done[k], cudaEventDisableTiming);
        }
    }
    if (e == cudaSuccess) e = cudaEventCreate(&f->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&f->ev1);
    if (e != cudaSuccess) {
        ggp_forest_destroy(f);
        return fail(e == cudaErrorMemoryAllocation ? GGP_ERR_NOMEM : GGP_ERR_CUDA,
                    std::string("forest upload: ") + cudaGetErrorString(e));
    }
    *out = f;
    return GGP_OK;
}

void ggp_forest_destroy(ggp_forest* f) {
    if (!f) return;
    cudaSetDevice(f->device);
    cudaDeviceSynchronize();
    for (DevBuf<double>* b : {&f->time, &f->x, &f->g, &f->w_params, &f->w_state, &f->w_partial, &f->w_out, &f->w_cell_ll,
                              &f->w_carry, &f->fwd, &f->bwd, &f->comb, &f->bstate, &f->pred_params, &f->prep, &f->jstack, &f->pack})
        b->release();
    for (DevBuf<int32_t>* b : {&f->seg, &f->comb_seg, &f->s_n, &f->s_parent, &f->s_d1, &f->s_d2, &f->s_root, &f->s_cell, &f->ctp_slot, &f->jstack_slot})
        b->release();
    f->s_off.release();
    f->s_dfs0.release();
    f->w_nan.release();
    f->w_invalid.release();
    f->dt_idx.release(); f->d_dt_values.release(); f->w_ktab.release();
    for (cudaEvent_t ev : f->chunk_ready) if (ev) cudaEventDestroy(ev);
    if (f->compute_done) cudaEventDestroy(f->compute_done);
    if (f->eval_start) cudaEventDestroy(f->eval_start);
    for (cudaEvent_t ev : f->chunk_done) if (ev) cudaEventDestroy(ev);
    for (cudaStream_t st : f->chunk_stream) if (st) cudaStreamDestroy(st);
    if (f->copy_stream) cudaStreamDestroy(f->copy_stream);
    for (cudaEvent_t ev : f->pass_done) if (ev) cudaEventDestroy(ev);
    if (f->ev0) cudaEventDestroy(f->ev0);
    if (f->ev1) cudaEventDestroy(f->ev1);
    delete f;
}

int ggp_forest_set_stream(ggp_forest* f, void* cuda_stream) {
    if (int rc = check_handle(f)) return rc;
    f->stream = (cudaStream_t)cuda_stream;
    return GGP_OK;
}

int ggp_forest_upload_series(ggp_forest* f, const double* time, const double* log_length, const double* fp,
                             const double* init_f4, const double* init_r4) {
    if (int rc = check_handle(f)) return rc;
    if (!time && !log_length && !fp) return fail(GGP_ERR_BAD_ARG, "no series given");
    if ((init_f4 == nullptr) != (init_r4 == nullptr)) return fail(GGP_ERR_BAD_ARG, "init_f4 and init_r4 go together");
    // the root / leaf priors are statistics of the CURRENT measurements (init_cells_f/r, moma_input.h:675-735)
    if (init_f4) {
        for (int i = 0; i < 4; ++i) { f->L.init_f[i] = init_f4[i]; f->L.init_r[i] = init_r4[i]; }
    } else if (log_length || fp) {
        if (!f->compute_init)
            return fail(GGP_ERR_BAD_ARG, "new measurements need their init_cells statistics: this forest was created with statistics of a "
                                         "larger data set (compute_init = 0), pass init_f4 / init_r4 (ggp_init_stats)");
        const int64_t N = f->n_cells;
        const std::vector<int64_t>& off = f->h_off;
        for (int64_t c = 0; c < N; ++c) {
            const int64_t o = off[c], l = off[c + 1] - 1;
            if (log_length) { f->edge[c] = log_length[o]; f->edge[N + c] = log_length[l]; }
            if (fp) { f->edge[2 * N + c] = fp[o]; f->edge[3 * N + c] = fp[l]; }
        }
        for (int dir = 0; dir < 2; ++dir) {   // GgpLayout::init_stats on the edge values: same sums in the same order
            double sx = 0, sg = 0, sxx = 0, sgg = 0;
            int64_t cnt = 0;
            const double* ex = f->edge.data() + (size_t)dir * N;
            const double* eg = f->edge.data() + (size_t)(2 + dir) * N;
            for (int64_t c = 0; c < N; ++c)
                if (off[c + 1] - off[c] > 1) {
                    sx += ex[c]; sg += eg[c]; sxx += ex[c] * ex[c]; sgg += eg[c] * eg[c];
                    ++cnt;
                }
            double* out = dir == 0 ? f->L.init_f : f->L.init_r;
            const double mx = sx / cnt, mg = sg / cnt;
            out[0] = mx; out[1] = mg; out[2] = sxx / cnt - mx * mx; out[3] = sgg / cnt - mg * mg;
        }
    }
    GGP_CUDA(cudaSetDevice(f->device));
    if (time) {   // a new time grid: the table of distinct time steps follows it (host pass; an unchanged grid should be passed as NULL)
        GGP_CUDA(cudaStreamSynchronize(f->stream));
        GGP_CUDA(build_dt_table(f, time));
    }
    // the copies run on their own stream, chunk by chunk, behind whatever the handle's stream still reads; the next
    // likelihood evaluation starts on a chunk's trees as soon as that chunk has landed (enqueue_loglik)
    GGP_CUDA(cudaEventRecord(f->compute_done, f->stream));
    GGP_CUDA(cudaStreamWaitEvent(f->copy_stream, f->compute_done, 0));
    for (int k = 0; k < f->L.n_chunks; ++k) {
        const int64_t c0 = f->L.ctp_chunk_start[k];
        const size_t b = (size_t)(f->L.ctp_chunk_start[k + 1] - c0) * sizeof(double);
        if (time) GGP_CUDA(cudaMemcpyAsync(f->time.p + c0, time + c0, b, cudaMemcpyHostToDevice, f->copy_stream));
        if (log_length) GGP_CUDA(cudaMemcpyAsync(f->x.p + c0, log_length + c0, b, cudaMemcpyHostToDevice, f->copy_stream));
        if (fp) GGP_CUDA(cudaMemcpyAsync(f->g.p + c0, fp + c0, b, cudaMemcpyHostToDevice, f->copy_stream));
        GGP_CUDA(cudaEventRecord(f->chunk_ready[k], f->copy_stream));
    }
    f->upload_pending = true;
    f->have_pred = false;
    f->have_prep = false;
    return GGP_OK;
}

int64_t ggp_forest_n_cells(const ggp_forest* f) { return f ? f->n_cells : -1; }
int64_t ggp_forest_n_ctp(const ggp_forest* f) { return f ? f->n_ctp : -1; }
int64_t ggp_forest_n_roots(const ggp_forest* f) { return f ? f->n_roots : -1; }
int64_t ggp_forest_n_generations(const ggp_forest* f) { return f ? f->n_gen : -1; }

int ggp_forest_get_init(const ggp_forest* f, double* init_f4, double* init_r4) {
    if (int rc = check_handle(f)) return rc;
    for (int i = 0; i < 4; ++i) {
        if (init_f4) init_f4[i] = f->L.init_f[i];
        if (init_r4) init_r4[i] = f->L.init_r[i];
    }
    return GGP_OK;
}

int ggp_init_stats(const ggp_forest_desc* d, double* init_f4, double* init_r4) {
    if (!d || !init_f4 || !init_r4 || d->n_cells <= 0 || !d->cell_offset || !d->log_length || !d->fp) return fail(GGP_ERR_BAD_ARG, "null argument");
    GgpLayout::init_stats(d, init_f4, init_r4);
    return GGP_OK;
}

int ggp_forest_set_mode(ggp_forest* f, int32_t mode) {
    if (int rc = check_handle(f)) return rc;
    if (mode == GGP_MODE_STRICT || mode == GGP_MODE_FAST || ggp_fast_supported_nodes(mode)) f->fast_mode = mode;
    else return fail(GGP_ERR_BAD_ARG, "unknown likelihood mode");
    return GGP_OK;
}
int32_t ggp_forest_get_mode(const ggp_forest* f) { return f ? f->fast_mode : -1; }
int32_t ggp_last_fast_nodes(const ggp_forest* f) { return f ? f->last_nodes : -1; }
int64_t ggp_last_strict_reruns(const ggp_forest* f) { return f ? f->last_reruns : -1; }

double ggp_last_kernel_ms(const ggp_forest* f) { return f ? f->last_ms : -1.0; }
int64_t ggp_last_launch_count(const ggp_forest* f) { return f ? f->last_launches : -1; }

}  // extern "C"

namespace {

// make the handle's stream wait for a pending streamed upload (all chunks)
int wait_for_upload(ggp_forest* f) {
    if (!f->upload_pending) return GGP_OK;
    for (cudaEvent_t ev : f->chunk_ready) GGP_CUDA(cudaStreamWaitEvent(f->stream, ev, 0));
    f->upload_pending = false;
    return GGP_OK;
}

// node counts of the fast kernels and the largest |d(exponent)/ds| * dt each rule integrates to rounding (GgpFastLmax)
const int kFastNodes[] = {4, 5, 6, 8, 10};
const double kFastLmax[] = {0.02, 0.12, 0.5, 1.8, 4.0};

// the smallest rule that covers a parameter vector on this forest: an a-priori bound of |b + lambda + C_xl| + gq + 4 a dt with
// lambda within three stationary standard deviations of its mean and a <= var_lambda / (4 gamma_lambda), times the largest
// time step, with a 10 % margin.  The kernels check the actual value at every step; a vector that still leaves the range is
// re-run with the next rule (then on the strict path).  0 = no rule covers it.
int pick_fast_nodes(const ggp_forest* f, const double* p) {
    const double sd_l = std::sqrt(std::fabs(p[2] / (2.0 * p[1])));
    const double lam = std::fabs(p[6]) + std::fabs(p[0]) + 3.0 * sd_l + std::fabs(p[4]) + std::fabs(p[2] / p[1]) * f->dt_max;
    const double need = 1.1 * lam * f->dt_max;
    if (!(need == need)) return 0;
    for (size_t i = 0; i < std::size(kFastNodes); ++i) if (need <= kFastLmax[i]) return kFastNodes[i];
    return 0;
}
int next_fast_nodes(int n) {
    for (size_t i = 0; i + 1 < std::size(kFastNodes); ++i) if (kFastNodes[i] == n) return kFastNodes[i + 1];
    return 0;
}

// the rule of a fresh-mode ggp_loglik (0 = the strict kernels): the handle's node count, or in mode 1 the smallest rule that
// covers every vector of the batch; if one vector has none, the whole batch runs on the strict kernels
int loglik_nodes(ggp_forest* f, const double* params, int32_t n_vec) {
    if (!f->dt_ok || f->fast_mode == 0) return 0;
    if (f->fast_mode > 1) return f->fast_mode;
    int nodes = kFastNodes[0];
    for (int32_t v = 0; v < n_vec && nodes; ++v) {
        const int nv = pick_fast_nodes(f, params + (size_t)v * GGP_NP);
        nodes = nv == 0 ? 0 : std::max(nodes, nv);
    }
    if (nodes) f->auto_nodes = f->last_nodes = nodes;
    return nodes;
}
// the rule of ggp_loglik_grad and ggp_loglik_hess in every mode: the handle's node count, else the smallest that covers every vector some rule covers
// a priori, the largest if no vector has one (the kernels check every step, the ladder takes it from there)
int grad_nodes(ggp_forest* f, const double* params, int32_t n_vec) {
    if (!f->dt_ok) return 0;
    int nodes = 0;
    if (f->fast_mode > 1) nodes = f->fast_mode;
    else {
        for (int32_t v = 0; v < n_vec; ++v) nodes = std::max(nodes, pick_fast_nodes(f, params + (size_t)v * GGP_NP));
        if (!nodes) nodes = kFastNodes[std::size(kFastNodes) - 1];
    }
    f->last_nodes = nodes;
    return nodes;
}

// enqueue the plan's evaluations of vectors [0, n_vec): parameters in d_params on the device, else h_params (at most
// GGP_INLINE_VECS vectors) travel in the launch arguments; every vector is evaluated plan.evals() times, with plan.comps()
// results each: d_out receives [n_vec][evals][comps] ([n_vec] for the log-likelihood, plan order 0).
// nodes > 0: the fast kernels with that rule (fresh mode only), which flag in w_invalid the vectors the caller has to re-run;
// nodes == 0: the strict kernels (order 0 only).  Derivatives run on the fast kernels from device parameters.
// The state of one vector chunk stays within the handle's budget: when one vector's evaluations exceed it, vectors go one at a
// time and their evaluations in ranges that fit (at least one evaluation per launch).  Every evaluation is independent, so
// chunking changes no bit as long as the launches partition each generation the same way (per_chunk below).
int enqueue_loglik(ggp_forest* f, int nodes, const double* d_params, const double* h_params, int32_t n_vec, double* d_carry,
                   const GgpEvalPlan& plan, double* d_out, double* d_cell_ll, unsigned long long* d_nan) {
    const int64_t N = f->n_cells;
    const int ne = plan.evals(), comps = plan.comps();
    const int64_t eval_bytes = N * 14 * comps * (int64_t)sizeof(double);
    int64_t chunk = f->state_budget_bytes / (eval_bytes * ne);
    int er = ne;   // evaluations of a vector per launch
    if (chunk < 1) {
        chunk = 1;
        er = (int)std::max<int64_t>(1, std::min<int64_t>(ne, f->state_budget_bytes / eval_bytes));
    }
    chunk = std::min<int64_t>(chunk, n_vec);
    chunk = std::min<int64_t>(chunk, 65535 / er);
    const int n_partial = f->n_partial;
    GGP_CUDA(f->w_state.ensure((size_t)chunk * er * N * 14 * comps));
    GGP_CUDA(f->w_partial.ensure((size_t)chunk * er * comps * n_partial));
    const GgpDevForest F = f->dev();
    const int K = f->L.n_chunks;
    // a freshly uploaded forest is evaluated chunk by chunk behind the copies (one launch sequence only; carry mode and
    // multi-chunk batches wait for the whole upload)
    const bool one_pass = chunk >= n_vec && er == ne;
    const bool streamed = f->upload_pending && K > 1 && !d_carry && one_pass;
    if (!d_params && !h_params) return fail(GGP_ERR_BAD_ARG, "inline parameters without a vector");
    if (nodes && d_carry) return fail(GGP_ERR_BAD_ARG, "the fast likelihood has no carry mode");
    if (plan.order && (!nodes || !d_params)) return fail(GGP_ERR_BAD_ARG, "derivatives run on the fast kernels from device parameters");
    if (!streamed) if (int rc = wait_for_upload(f)) return rc;
    for (int32_t v0 = 0; v0 < n_vec; v0 += (int32_t)chunk)
    for (int e0 = 0; e0 < ne; e0 += er) {
        const int32_t vc = (int32_t)std::min<int64_t>(chunk, n_vec - v0);
        const int ec = std::min(er, ne - e0);   // er < ne only with vc == 1: the outputs of a launch are contiguous
        GgpEvalPlan run = plan;
        run.select(e0, ec);
        // launches do not write every partial (whole-generation launches pack their groups)
        {
            const size_t cnt = (size_t)vc * ec * comps * n_partial;
            ggp_fill64_kernel<<<f->fill_grid(cnt), 256, 0, f->stream>>>(reinterpret_cast<unsigned long long*>(f->w_partial.p), 0ull, cnt);
        }
        if (nodes) {   // the (parameters, dt)-only constants of this vector chunk
            GGP_CUDA(f->w_ktab.ensure((size_t)vc * ec * f->dt_values.size() * ggp_fast_consts_bytes(run, nodes)));
            GgpFwdArgs C{};
            C.params = d_params;
            if (!d_params) std::memcpy(C.inline_params, h_params, (size_t)n_vec * GGP_NP * sizeof(double));
            C.v0 = v0;
            C.v_count = vc;
            GGP_CUDA(ggp_fast_consts_launch(C, run, f->d_dt_values.p, (int)f->dt_values.size(), f->w_ktab.p, nodes, f->stream));
            ++f->last_launches;
        }
        // per_chunk: the forest's upload chunks (groups of whole trees) are evaluated one after the other, each on a stream of
        // its own, so that the few-block early generations of one chunk run beside the large late generations of another.
        // Always behind a streamed upload; for the fast kernels (128-thread blocks, two per SM, no shared-memory footprint:
        // launches of different streams share the SMs) also on a resident forest, the likelihood and the gradient when the batch
        // is one vector chunk, the Hessian always: the launches partition a generation into blocks (and partial sums)
        // differently, and the Hessian's bits must not depend on how the state budget splits its evaluations.
        const bool per_chunk = streamed || (nodes && K > 1 && (chunk >= n_vec || plan.order == 2));
        if (per_chunk) GGP_CUDA(cudaEventRecord(f->eval_start, f->stream));
        for (int k = 0; k < (per_chunk ? K : 1); ++k) {
            // stream of this chunk's launches: its own (behind everything enqueued on the handle's stream so far), the
            // handle's for the last chunk
            const cudaStream_t ks = (per_chunk && k + 1 < K) ? f->chunk_stream[k] : f->stream;
            if (per_chunk && k + 1 < K) GGP_CUDA(cudaStreamWaitEvent(ks, f->eval_start, 0));
            if (streamed) GGP_CUDA(cudaStreamWaitEvent(ks, f->chunk_ready[k], 0));
            for (int g = 0; g < f->n_gen; ++g) {
                const int64_t* row = f->L.gen_chunk_start.data() + (size_t)g * (K + 1);
                GgpFwdArgs A{};
                A.slot0 = (int)(per_chunk ? row[k] : row[0]);
                A.n_slots = (int)((per_chunk ? row[k + 1] : row[K]) - A.slot0);
                if (A.n_slots == 0) continue;
                A.params = d_params;
                if (!d_params) std::memcpy(A.inline_params, h_params, (size_t)n_vec * GGP_NP * sizeof(double));
                A.v0 = v0;
                A.v_count = vc;
                A.carry = d_carry;
                A.state = f->w_state.p;
                A.partial = f->w_partial.p;
                A.partial0 = f->gen_partial0[(size_t)g * (K + 1) + (per_chunk ? k : 0)];
                A.n_partial = n_partial;
                A.cell_ll = d_cell_ll;
                A.nan_key = d_nan;
                A.out_fwd = nullptr;
                const int ng = grid_of_coop(A.n_slots);
                if (nodes)
                    GGP_CUDA(ggp_fast_loglik_launch(F, A, run, f->w_ktab.p, f->w_invalid.p, nodes, ks));
                else if (g == 0 && d_carry)
                    ggp_loglik_chain_coop_kernel<<<dim3(ng, 1), GGP_COOP_BLOCK(1), GGP_COOP_SMEM_BYTES_CHAIN, ks>>>(F, A);
                else if ((int64_t)ng * vc >= f->coop_ng4_min_groups)
                    ggp_loglik_coop_kernel<4><<<dim3((ng + 3) / 4, vc), GGP_COOP_BLOCK(4), GGP_COOP_SMEM_BYTES(4), ks>>>(F, A);
                else
                    ggp_loglik_coop_kernel<1><<<dim3(ng, vc), GGP_COOP_BLOCK(1), GGP_COOP_SMEM_BYTES(1), ks>>>(F, A);
                ++f->last_launches;
            }
            if (per_chunk && k + 1 < K) GGP_CUDA(cudaEventRecord(f->chunk_done[k], ks));
        }
        if (per_chunk) for (int k = 0; k + 1 < K; ++k) GGP_CUDA(cudaStreamWaitEvent(f->stream, f->chunk_done[k], 0));
        ggp_reduce_kernel<<<vc * ec * comps, 256, 0, f->stream>>>(f->w_partial.p, n_partial, d_out + ((size_t)v0 * ne + e0) * comps);
        ++f->last_launches;
    }
    if (streamed) f->upload_pending = false;
    GGP_CUDA(cudaGetLastError());
    return GGP_OK;
}

// the prologue of an evaluation on the handle's stream: the NaN keys (with_keys, w_nan) and the fast kernels' flags (nodes > 0,
// w_invalid) are cleared, then enqueue_loglik runs between ev0 and ev1
int enqueue_pass(ggp_forest* f, int nodes, const double* d_params, const double* h_params, int32_t n_vec, double* d_carry,
                 const GgpEvalPlan& plan, double* d_out, double* d_cell_ll, bool with_keys) {
    cudaStream_t s = f->stream;
    if (with_keys) {
        GGP_CUDA(f->w_nan.ensure(n_vec));
        ggp_fill64_kernel<<<f->fill_grid((size_t)n_vec), 256, 0, s>>>(f->w_nan.p, ~0ull, (size_t)n_vec);
    }
    if (nodes) {   // cleared by a kernel: a memset may queue behind a streamed upload's copies
        GGP_CUDA(f->w_invalid.ensure((size_t)n_vec + 1));
        ggp_fill64_kernel<<<f->fill_grid(((size_t)n_vec + 1) / 2), 256, 0, s>>>(reinterpret_cast<unsigned long long*>(f->w_invalid.p), 0ull, ((size_t)n_vec + 1) / 2);
    }
    GGP_CUDA(cudaEventRecord(f->ev0, s));
    if (int rc = enqueue_loglik(f, nodes, d_params, h_params, n_vec, d_carry, plan, d_out, d_cell_ll, with_keys ? f->w_nan.p : nullptr))
        return rc;
    GGP_CUDA(cudaEventRecord(f->ev1, s));
    return GGP_OK;
}

// one evaluation of the host vectors params [0, n_vec) with the rule `nodes` (0 = the strict kernels), returned when its results
// are on the host: out [n_vec][evals][comps] of the plan and, where the pointers are given, the
// NaN keys [n_vec], the fast kernels' flags [n_vec] and the per-cell rows [n_vec][n_cells]; carry [n_roots][16] is updated in
// place.  Adds its device time to last_ms (and enqueue_loglik its launches to last_launches).
int run_pass(ggp_forest* f, int nodes, const double* params, int32_t n_vec, double* carry, const GgpEvalPlan& plan, double* out,
             unsigned long long* keys, int* invalid, double* cell_ll) {
    cudaStream_t s = f->stream;
    const size_t n_out = (size_t)n_vec * plan.evals() * plan.comps();
    GGP_CUDA(f->w_params.ensure((size_t)n_vec * GGP_NP));
    GGP_CUDA(f->w_out.ensure(n_out));
    if (cell_ll) GGP_CUDA(f->w_cell_ll.ensure((size_t)n_vec * f->n_cells));
    if (carry) {
        GGP_CUDA(f->w_carry.ensure((size_t)f->n_roots * 16));
        GGP_CUDA(cudaMemcpyAsync(f->w_carry.p, carry, (size_t)f->n_roots * 16 * sizeof(double), cudaMemcpyHostToDevice, s));
    }
    // derivatives wait for the whole pending upload.  Behind a streamed upload a DMA copy of the parameters would queue after
    // the whole upload in the host-to-device copy engine: small batches travel in the launch arguments instead
    if (plan.order) if (int rc = wait_for_upload(f)) return rc;
    const bool inline_params = n_vec <= GGP_INLINE_VECS && f->upload_pending && !carry;
    if (!inline_params)
        GGP_CUDA(cudaMemcpyAsync(f->w_params.p, params, (size_t)n_vec * GGP_NP * sizeof(double), cudaMemcpyHostToDevice, s));
    if (int rc = enqueue_pass(f, nodes, inline_params ? nullptr : f->w_params.p, params, n_vec, carry ? f->w_carry.p : nullptr, plan,
                              f->w_out.p, cell_ll ? f->w_cell_ll.p : nullptr, keys != nullptr))
        return rc;
    GGP_CUDA(cudaMemcpyAsync(out, f->w_out.p, n_out * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (keys) GGP_CUDA(cudaMemcpyAsync(keys, f->w_nan.p, (size_t)n_vec * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    if (invalid) GGP_CUDA(cudaMemcpyAsync(invalid, f->w_invalid.p, (size_t)n_vec * sizeof(int), cudaMemcpyDeviceToHost, s));
    if (cell_ll) GGP_CUDA(cudaMemcpyAsync(cell_ll, f->w_cell_ll.p, (size_t)n_vec * f->n_cells * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (carry) GGP_CUDA(cudaMemcpyAsync(carry, f->w_carry.p, (size_t)f->n_roots * 16 * sizeof(double), cudaMemcpyDeviceToHost, s));
    GGP_CUDA(cudaStreamSynchronize(s));
    float ms = 0.f;
    GGP_CUDA(cudaEventElapsedTime(&ms, f->ev0, f->ev1));
    f->last_ms += ms;
    return GGP_OK;
}

// the re-run ladder of an evaluation of the host vectors params [0, n_vec): all of them with the rule `nodes`, the vectors a
// rule flags (they left its validity range or met a NaN term) with the next larger rule, what the largest rule flags with the
// strict kernels (rule 0: no flags, no derivatives).  Every pass puts the value, gradient row and Hessian block (the plan D's
// derivatives, natural space: GgpEvalPlan::unscale undoes the polarization of order 2), per-cell row and NaN record of the vectors it accepts
// into the caller's rows.  The first pass reads the caller's params and, without derivatives, writes ll and cell_ll in place;
// the others evaluate a compacted copy of the flagged vectors.  left: the vectors that went on from a fast pass to the strict
// kernels (their derivative rows are not written).  Sets the handle's counters; returns GGP_ERR_NAN if a NaN record was written.
int ladder(ggp_forest* f, int nodes, const double* params, int32_t n_vec, double* carry, const GgpEvalPlan& D, double* ll, double* grad,
           double* hess, double* cell_ll, ggp_nan_info* nan, std::vector<int32_t>& left) {
    const size_t N = (size_t)f->n_cells;
    std::vector<unsigned long long> keys((size_t)n_vec, ~0ull);   // the gradient kernels write no keys
    std::vector<int> invalid(nodes ? (size_t)n_vec : 0);
    std::vector<double> P, out, cl;
    std::vector<int32_t> flagged;
    bool any_nan = false;
    f->last_ms = 0.0;
    f->last_launches = 0;
    left.clear();
    for (int n = nodes, first = 1;; n = next_fast_nodes(n), first = 0) {
        const int32_t m = first ? n_vec : (int32_t)left.size();
        const GgpEvalPlan g = n ? D : GgpEvalPlan{};   // the strict kernels: the log-likelihood
        const size_t stride = (size_t)g.evals() * g.comps();
        const bool direct = first && !g.order;
        if (!first) {
            P.resize((size_t)m * GGP_NP);
            for (int32_t i = 0; i < m; ++i) std::memcpy(&P[(size_t)i * GGP_NP], params + (size_t)left[i] * GGP_NP, GGP_NP * sizeof(double));
        }
        if (!direct) {
            out.resize(m * stride);
            cl.resize(cell_ll ? m * N : 0);
        }
        if (int rc = run_pass(f, n, first ? params : P.data(), m, carry, g, direct ? ll : out.data(), g.order ? nullptr : keys.data(),
                              n ? invalid.data() : nullptr, !cell_ll ? nullptr : direct ? cell_ll : cl.data()))
            return rc;
        flagged.clear();
        for (int32_t i = 0; i < m; ++i) {
            const int32_t v = first ? i : left[i];
            if (n && invalid[i]) {
                flagged.push_back(v);
                continue;
            }
            int64_t cell = -1, t = -1;
            if (keys[i] != ~0ull) {
                any_nan = true;
                f->L.locate((int64_t)keys[i], &cell, &t);
            }
            if (nan) { nan[v].cell = cell; nan[v].t_index = t; }
            if (direct) continue;
            const double* o = &out[i * stride];
            ll[v] = o[0];   // every evaluation carries the same value: the first one's
            if (g.order) g.unscale(params + (size_t)v * GGP_NP, o, grad + (size_t)v * g.n_dirs, hess ? hess + (size_t)v * g.n_dirs * g.n_dirs : nullptr);
            if (cell_ll) std::memcpy(cell_ll + v * N, &cl[i * N], N * sizeof(double));
        }
        if (!n) break;
        left.swap(flagged);
        if (left.empty()) break;
    }
    f->last_reruns = (int64_t)left.size();
    return any_nan ? fail(GGP_ERR_NAN, "Likelihood is Nan") : GGP_OK;
}

}  // namespace

extern "C" {

int ggp_loglik(ggp_forest* f, const double* params, int32_t n_vec, double* root_carry, double* out_loglik,
               double* out_cell_ll, ggp_nan_info* nan) {
    if (int rc = check_handle(f)) return rc;
    if (!params || !out_loglik || n_vec <= 0) return fail(GGP_ERR_BAD_ARG, "bad params/out/n_vec");
    GGP_CUDA(cudaSetDevice(f->device));
    std::vector<int32_t> left;
    return ladder(f, root_carry ? 0 : loglik_nodes(f, params, n_vec), params, n_vec, root_carry, GgpEvalPlan{}, out_loglik, nullptr, nullptr,
                  out_cell_ll, nan, left);
}

int ggp_loglik_device(ggp_forest* f, const double* d_params, int32_t n_vec, double* d_out_loglik) {
    if (int rc = check_handle(f)) return rc;
    if (!d_params || !d_out_loglik || n_vec <= 0) return fail(GGP_ERR_BAD_ARG, "bad params/out/n_vec");
    GGP_CUDA(cudaSetDevice(f->device));
    const int nodes = !f->dt_ok ? 0 : (f->fast_mode > 1 ? f->fast_mode : (f->fast_mode == 1 ? f->auto_nodes : 0));
    f->last_launches = 0;
    f->device_fast_vecs = nodes ? n_vec : 0;   // the flags are checked by ggp_sync_kernel_ms
    return enqueue_pass(f, nodes, d_params, nullptr, n_vec, nullptr, GgpEvalPlan{}, d_out_loglik, nullptr, true);
}

}  // extern "C"

namespace {

// the directions of a gradient call: NULL = all GGP_NP parameters (n_dirs = GGP_NP), else distinct indices 0 .. GGP_NP - 1
int grad_dirs(const int32_t* dirs, int32_t n_dirs, GgpEvalPlan& P) {
    if (!dirs) {
        if (n_dirs != GGP_NP) return fail(GGP_ERR_BAD_ARG, "dirs = NULL differentiates all 11 parameters: n_dirs must be 11");
        P.n_dirs = GGP_NP;
        for (int i = 0; i < GGP_NP; ++i) P.dirs[i] = i;
        return GGP_OK;
    }
    if (n_dirs <= 0 || n_dirs > GGP_NP) return fail(GGP_ERR_BAD_ARG, "n_dirs must be 1 .. 11");
    bool seen[GGP_NP] = {};
    for (int32_t i = 0; i < n_dirs; ++i) {
        const int32_t d = dirs[i];
        if (d < 0 || d >= GGP_NP) return fail(GGP_ERR_BAD_ARG, "dirs[" + std::to_string(i) + "] = " + std::to_string(d) + " is not a parameter index (0 .. 10)");
        if (seen[d]) return fail(GGP_ERR_BAD_ARG, "parameter index " + std::to_string(d) + " appears twice in dirs");
        seen[d] = true;
        P.dirs[i] = d;
    }
    P.n_dirs = n_dirs;
    return GGP_OK;
}

// ggp_loglik_grad (order 1) and ggp_loglik_hess (order 2, out_hess [n_vec][n_dirs][n_dirs])
int loglik_derivs(ggp_forest* f, int order, const double* params, int32_t n_vec, const int32_t* dirs, int32_t n_dirs, double* out_loglik,
                  double* out_grad, double* out_hess, ggp_nan_info* nan) {
    if (int rc = check_handle(f)) return rc;
    if (!params || !out_loglik || !out_grad || (order == 2 && !out_hess) || n_vec <= 0) return fail(GGP_ERR_BAD_ARG, "bad params/out/n_vec");
    GgpEvalPlan D{};
    D.order = order;
    if (int rc = grad_dirs(dirs, n_dirs, D)) return rc;
    GGP_CUDA(cudaSetDevice(f->device));
    const int nodes = grad_nodes(f, params, n_vec);
    std::vector<ggp_nan_info> own(nan ? 0 : (size_t)n_vec);
    ggp_nan_info* rec = nan ? nan : own.data();
    std::vector<int32_t> left;
    const int rc = ladder(f, nodes, params, n_vec, nullptr, D, out_loglik, out_grad, out_hess, nullptr, rec, left);
    if (rc != GGP_OK && rc != GGP_ERR_NAN) return rc;
    if (!nodes) {   // no rule without the table of time steps: every vector went to the strict kernels
        left.resize((size_t)n_vec);
        std::iota(left.begin(), left.end(), 0);
        f->last_reruns = n_vec;
    }
    if (left.empty()) return GGP_OK;
    // what no rule covers, or what meets a NaN term: the strict value (and NaN record), NaN derivative rows
    const int32_t n = D.n_dirs;
    std::string uncovered;
    for (int32_t v : left) {
        for (int32_t j = 0; j < n; ++j) out_grad[(size_t)v * n + j] = std::nan("");
        if (out_hess) for (int32_t j = 0; j < n * n; ++j) out_hess[(size_t)v * n * n + j] = std::nan("");
        if (rec[v].cell < 0) uncovered += (uncovered.empty() ? "" : ", ") + std::to_string(v);
    }
    if (!uncovered.empty())
        return fail(GGP_ERR_BAD_ARG, std::string(order == 1 ? "fast gradient" : "fast Hessian") +
                                         ": no quadrature rule covers parameter vector(s) " + uncovered + " (log-likelihood: the strict value; " +
                                         (order == 1 ? "gradient row: NaN)" : "gradient and Hessian rows: NaN)"));
    return fail(GGP_ERR_NAN, "Likelihood is Nan");
}

}  // namespace

extern "C" {

int ggp_loglik_grad(ggp_forest* f, const double* params, int32_t n_vec, const int32_t* dirs, int32_t n_dirs, double* out_loglik,
                    double* out_grad, ggp_nan_info* nan) {
    return loglik_derivs(f, 1, params, n_vec, dirs, n_dirs, out_loglik, out_grad, nullptr, nan);
}

int ggp_loglik_hess(ggp_forest* f, const double* params, int32_t n_vec, const int32_t* dirs, int32_t n_dirs, double* out_loglik,
                    double* out_grad, double* out_hess, ggp_nan_info* nan) {
    return loglik_derivs(f, 2, params, n_vec, dirs, n_dirs, out_loglik, out_grad, out_hess, nan);
}

int ggp_sync_kernel_ms(ggp_forest* f, double* ms_out) {
    if (int rc = check_handle(f)) return rc;
    GGP_CUDA(cudaSetDevice(f->device));
    GGP_CUDA(cudaEventSynchronize(f->ev1));
    float ms = 0.f;
    GGP_CUDA(cudaEventElapsedTime(&ms, f->ev0, f->ev1));
    f->last_ms = ms;
    if (ms_out) *ms_out = ms;
    if (f->device_fast_vecs > 0) {   // a fast evaluation enqueued by ggp_loglik_device: was every vector inside the validity range?
        std::vector<int> invalid((size_t)f->device_fast_vecs);
        GGP_CUDA(cudaMemcpy(invalid.data(), f->w_invalid.p, invalid.size() * sizeof(int), cudaMemcpyDeviceToHost));
        f->device_fast_vecs = 0;
        for (int v : invalid)
            if (v) return fail(GGP_ERR_BAD_ARG, "fast likelihood: a parameter vector left the quadrature's validity range; evaluate it with ggp_loglik (which re-runs it strictly)");
    }
    return GGP_OK;
}

}  // extern "C"

namespace {

// [n][20] (4 means + row-major 4x4) -> [n][14] (4 means + upper triangle row-major: xx xg xl xq gg gl gq ll lq qq), the 14
// numbers per time point the reference's writer prints (predictions.h:541-552, 575-578)
__global__ void __launch_bounds__(256) ggp_pack14_kernel(int64_t n, const double* __restrict__ in20, double* __restrict__ out14) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n * 14) return;
    const int64_t k = i / 14;
    const int e = (int)(i - k * 14);
    constexpr int src[14] = {0, 1, 2, 3, 4, 5, 6, 7, 9, 10, 11, 14, 15, 19};
    out14[i] = in20[20 * k + src[e]];
}

int predict_impl(ggp_forest* f, const double* params, int32_t n_seg, double* out_forward, double* out_backward,
                 double* out_combined, bool pack14) {
    if (int rc = check_handle(f)) return rc;
    if (!params || n_seg <= 0) return fail(GGP_ERR_BAD_ARG, "bad params/n_seg");
    if (f->max_seg >= n_seg) return fail(GGP_ERR_BAD_ARG, "segment index exceeds the number of parameter sets");
    GGP_CUDA(cudaSetDevice(f->device));
    cudaStream_t s = f->stream;
    const int64_t N = f->n_cells, M = f->n_ctp;
    GGP_CUDA(f->pred_params.ensure((size_t)n_seg * GGP_NP));
    GGP_CUDA(f->w_state.ensure((size_t)N * 14));
    GGP_CUDA(f->fwd.ensure((size_t)M * 20));
    GGP_CUDA(f->bwd.ensure((size_t)M * 20));
    GGP_CUDA(f->comb.ensure((size_t)M * 20));
    GGP_CUDA(f->bstate.ensure((size_t)N * 20));
    GGP_CUDA(cudaMemcpyAsync(f->pred_params.p, params, (size_t)n_seg * GGP_NP * sizeof(double), cudaMemcpyHostToDevice, s));
    if (int rc = wait_for_upload(f)) return rc;
    f->pred_n_seg = n_seg;
    f->have_pred = false;
    f->have_prep = false;
    f->last_launches = 0;
    const GgpDevForest F = f->dev();
    // an output leaves for the host as soon as its pass has finished, on the copy stream, while the next pass runs (the copies
    // are 6 x the kernels on configs[2]); pack14: 30 % fewer bytes across PCIe, packed on the device into one staging buffer per output
    const double* src[3] = {f->fwd.p, f->bwd.p, f->comb.p};
    double* dst[3] = {out_forward, out_backward, out_combined};
    if (pack14) {
        int n_out = 0;
        for (int o = 0; o < 3; ++o) n_out += dst[o] != nullptr;
        GGP_CUDA(f->pack.ensure((size_t)M * 14 * std::max(n_out, 1)));
    }
    int pack_slot = 0;
    auto ship = [&](int o) -> int {
        if (!dst[o]) return GGP_OK;
        GGP_CUDA(cudaEventRecord(f->pass_done[o], s));
        GGP_CUDA(cudaStreamWaitEvent(f->copy_stream, f->pass_done[o], 0));
        if (pack14) {
            double* stage = f->pack.p + (size_t)M * 14 * pack_slot++;
            ggp_pack14_kernel<<<(unsigned)((M * 14 + 255) / 256), 256, 0, f->copy_stream>>>(M, src[o], stage);
            GGP_CUDA(cudaMemcpyAsync(dst[o], stage, (size_t)M * 14 * sizeof(double), cudaMemcpyDeviceToHost, f->copy_stream));
        } else {
            GGP_CUDA(cudaMemcpyAsync(dst[o], src[o], (size_t)M * 20 * sizeof(double), cudaMemcpyDeviceToHost, f->copy_stream));
        }
        return GGP_OK;
    };
    GGP_CUDA(cudaEventRecord(f->ev0, s));
    for (int g = 0; g < f->n_gen; ++g) {
        GgpFwdArgs A{};
        A.slot0 = (int)f->L.gen_start[g];
        A.n_slots = (int)(f->L.gen_start[g + 1] - f->L.gen_start[g]);
        A.params = f->pred_params.p;
        A.v0 = 0;
        A.v_count = 1;
        A.state = f->w_state.p;
        A.out_fwd = f->fwd.p;
        A.n_seg = n_seg;
        const int ng = grid_of_coop(A.n_slots);
        if (ng >= f->coop_ng4_min_groups && n_seg == 1)
            ggp_loglik_coop_kernel<kPredUniNG, true, true><<<dim3((ng + kPredUniNG - 1) / kPredUniNG, 1), GGP_COOP_BLOCK(kPredUniNG), GGP_COOP_SMEM_BYTES(kPredUniNG), s>>>(F, A);
        else if (ng >= f->coop_ng4_min_groups)
            ggp_loglik_coop_kernel<kPredNG, true><<<dim3((ng + kPredNG - 1) / kPredNG, 1), GGP_COOP_BLOCK(kPredNG), GGP_COOP_SMEM_BYTES(kPredNG), s>>>(F, A);
        else
            ggp_loglik_coop_kernel<1, true><<<dim3(ng, 1), GGP_COOP_BLOCK(1), GGP_COOP_SMEM_BYTES(1), s>>>(F, A);
        ++f->last_launches;
    }
    if (int rc = ship(0)) return rc;
    for (int g = f->n_gen - 1; g >= 0; --g) {
        GgpBwdArgs B{};
        B.slot0 = (int)f->L.gen_start[g];
        B.n_slots = (int)(f->L.gen_start[g + 1] - f->L.gen_start[g]);
        B.params = f->pred_params.p;
        B.fwd = f->fwd.p;
        B.bwd = f->bwd.p;
        B.bstate = f->bstate.p;
        B.n_seg = n_seg;
        const int ng = grid_of_coop(B.n_slots);
        if (ng >= f->coop_ng4_min_groups && n_seg == 1)
            ggp_backward_coop_kernel<kPredUniNG, true><<<(ng + kPredUniNG - 1) / kPredUniNG, GGP_COOP_BLOCK(kPredUniNG), GGP_COOP_SMEM_BYTES(kPredUniNG), s>>>(F, B);
        else if (ng >= f->coop_ng4_min_groups)
            ggp_backward_coop_kernel<kPredNG><<<(ng + kPredNG - 1) / kPredNG, GGP_COOP_BLOCK(kPredNG), GGP_COOP_SMEM_BYTES(kPredNG), s>>>(F, B);
        else
            ggp_backward_coop_kernel<1><<<ng, GGP_COOP_BLOCK(1), GGP_COOP_SMEM_BYTES(1), s>>>(F, B);
        ++f->last_launches;
    }
    if (int rc = ship(1)) return rc;
    ggp_combine_kernel<<<grid_of(M), GGP_BLOCK, 0, s>>>(M, f->fwd.p, f->bwd.p, f->comb_seg.p, f->pred_params.p, f->comb.p);
    ++f->last_launches;
    GGP_CUDA(cudaGetLastError());
    GGP_CUDA(cudaEventRecord(f->ev1, s));
    if (int rc = ship(2)) return rc;
    GGP_CUDA(cudaStreamSynchronize(f->copy_stream));
    GGP_CUDA(cudaStreamSynchronize(s));
    float ms = 0.f;
    GGP_CUDA(cudaEventElapsedTime(&ms, f->ev0, f->ev1));
    f->last_ms = ms;
    f->have_pred = true;
    return GGP_OK;
}

}  // namespace

extern "C" {

int ggp_predict(ggp_forest* f, const double* params, int32_t n_seg, double* out_forward, double* out_backward,
                double* out_combined) {
    return predict_impl(f, params, n_seg, out_forward, out_backward, out_combined, false);
}

int ggp_predict14(ggp_forest* f, const double* params, int32_t n_seg, double* out_forward14, double* out_backward14,
                  double* out_combined14) {
    return predict_impl(f, params, n_seg, out_forward14, out_backward14, out_combined14, true);
}

int ggp_backward_cell_state(ggp_forest* f, double* out_cell_state20) {
    if (int rc = check_handle(f)) return rc;
    if (!f->have_pred) return fail(GGP_ERR_BAD_ARG, "ggp_predict has not been run on this handle");
    if (!out_cell_state20) return fail(GGP_ERR_BAD_ARG, "null output");
    GGP_CUDA(cudaSetDevice(f->device));
    std::vector<double> tmp((size_t)f->n_cells * 20);
    GGP_CUDA(cudaMemcpyAsync(tmp.data(), f->bstate.p, tmp.size() * sizeof(double), cudaMemcpyDeviceToHost, f->stream));
    GGP_CUDA(cudaStreamSynchronize(f->stream));
    for (int64_t s = 0; s < f->n_cells; ++s)
        std::memcpy(out_cell_state20 + 20 * (int64_t)f->L.cell_of_slot[s], tmp.data() + 20 * s, 20 * sizeof(double));
    return GGP_OK;
}

int ggp_math_eval(int32_t device, int32_t fn, int64_t n, const double* x, const double* y, double* out) {
    if (!x || !out || n <= 0 || fn < 0 || fn > 6 || ((fn == 2 || fn == 4 || fn == 5) && !y)) return fail(GGP_ERR_BAD_ARG, "bad argument");
    GGP_CUDA(cudaSetDevice(device));
    const int64_t nx = fn == 6 ? 5 * n : n, nout = fn == 5 ? 5 * n : n;   // fn 6 reads five doubles per case, fn 5 writes five
    DevBuf<double> dx, dy, dout;
    GGP_CUDA(dx.ensure(nx));
    GGP_CUDA(dy.ensure(n));
    GGP_CUDA(dout.ensure(nout));
    GGP_CUDA(cudaMemcpy(dx.p, x, nx * sizeof(double), cudaMemcpyHostToDevice));
    if (y) GGP_CUDA(cudaMemcpy(dy.p, y, n * sizeof(double), cudaMemcpyHostToDevice));
    if (fn >= 5) {
        GGP_CUDA(opt_in_smem());
        ggp_coop_math_kernel<<<(unsigned)((n + GGP_COOP_CELLS - 1) / GGP_COOP_CELLS), GGP_COOP_CELLS, GGP_COOP_SMEM_BYTES(1)>>>(fn, n, dx.p, dy.p, dout.p);
    } else {
        ggp_math_kernel<<<grid_of(n), GGP_BLOCK, sizeof(GgpMathTables)>>>(fn, n, dx.p, dy.p, dout.p);
    }
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaMemcpy(out, dout.p, nout * sizeof(double), cudaMemcpyDeviceToHost);
    dx.release(); dy.release(); dout.release();
    if (e != cudaSuccess) return fail(GGP_ERR_CUDA, cudaGetErrorString(e));
    return GGP_OK;
}

int ggp_propagate_eval(int32_t device, int64_t n, const double* state14, const double* dt, const double* p7,
                       double* out14, double* cross16) {
    if (!state14 || !dt || !p7 || !out14 || n <= 0) return fail(GGP_ERR_BAD_ARG, "bad argument");
    GGP_CUDA(cudaSetDevice(device));
    DevBuf<double> ds, dd, dp, dout, dc;
    GGP_CUDA(ds.ensure(14 * n));
    GGP_CUDA(dd.ensure(n));
    GGP_CUDA(dp.ensure(7 * n));
    GGP_CUDA(dout.ensure(14 * n));
    if (cross16) GGP_CUDA(dc.ensure(16 * n));
    GGP_CUDA(cudaMemcpy(ds.p, state14, 14 * n * sizeof(double), cudaMemcpyHostToDevice));
    GGP_CUDA(cudaMemcpy(dd.p, dt, n * sizeof(double), cudaMemcpyHostToDevice));
    GGP_CUDA(cudaMemcpy(dp.p, p7, 7 * n * sizeof(double), cudaMemcpyHostToDevice));
    GGP_CUDA(opt_in_smem());
    ggp_propagate_kernel<<<grid_of(n), GGP_BLOCK, GGP_SMEM_BYTES>>>(n, ds.p, dd.p, dp.p, dout.p, cross16 ? dc.p : nullptr);
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaMemcpy(out14, dout.p, 14 * n * sizeof(double), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && cross16) e = cudaMemcpy(cross16, dc.p, 16 * n * sizeof(double), cudaMemcpyDeviceToHost);
    ds.release(); dd.release(); dp.release(); dout.release(); dc.release();
    if (e != cudaSuccess) return fail(GGP_ERR_CUDA, cudaGetErrorString(e));
    return GGP_OK;
}

int ggp_fp64_peak(int32_t device, double* tflops_out) {
    if (!tflops_out) return fail(GGP_ERR_BAD_ARG, "null output");
    GGP_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    GGP_CUDA(cudaGetDeviceProperties(&prop, device));
    DevBuf<double> out;
    GGP_CUDA(out.ensure(1));
    ScopedEvent e0, e1;   // destroyed on every return path
    GGP_CUDA(e0.create());
    GGP_CUDA(e1.create());
    const int blocks = prop.multiProcessorCount * 8, iters = 1 << 15;
    double best = 0.0;
    for (int rep = 0; rep < 6; ++rep) {
        GGP_CUDA(cudaEventRecord(e0.ev));
        ggp_fp64_peak_kernel<<<blocks, 256>>>(iters, 0.999999, 1e-9, out.p);
        GGP_CUDA(cudaEventRecord(e1.ev));
        GGP_CUDA(cudaEventSynchronize(e1.ev));
        float ms = 0.f;
        GGP_CUDA(cudaEventElapsedTime(&ms, e0.ev, e1.ev));
        const double tf = 2.0 * 8.0 * (double)iters * 256.0 * blocks / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    out.release();
    *tflops_out = best;
    return GGP_OK;
}

#ifdef GGP_PHASE_CLOCKS
// profiling builds only: out[role][10] = clocks per (phase work / barrier wait) slot, see ggp_coop_kernels.cuh
int ggp_debug_phase_clocks(unsigned long long* out, int reset) {
    if (out) GGP_CUDA(cudaMemcpyFromSymbol(out, ggp_phase_clk, sizeof(ggp_phase_clk)));
    if (reset) {
        unsigned long long z[GGP_COOP_ROLES][10] = {};
        GGP_CUDA(cudaMemcpyToSymbol(ggp_phase_clk, z, sizeof(z)));
    }
    return GGP_OK;
}
#endif

}  // extern "C"

#include "ggp_joints_host.inc"
#include "ggp_corr.inc"
#include "ggp_group.inc"
