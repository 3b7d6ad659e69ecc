// ggp_coop_kernels.cuh — lineage-forest passes with the four-warps-per-32-cells step of ggp_coop.cuh.
//
// Replaces, from the reference (paths under src/): likelihood_recr / total_likelihood (likelihood.h:110-174),
// prediction_forward / prediction_backward (predictions.h:166, 438).
// One launch per generation (y = parameter vector); a group of 128 threads owns 32 cells: lane = cell, warp = role.
// See ggp_coop.cuh for the phase plan.
#pragma once
#include "ggp_kernels.cuh"
#include "ggp_coop.cuh"

// A block holds NG groups of four warps (32 cells each) that share one copy of the math tables.  Warp w has role w % 4
// (so the four warps of one scheduler run the same role's instruction stream at about the same time: one instruction
// fetch serves NG groups) and group w / 4.
//   NG = 1: 128 threads, 4 blocks per SM; finest granularity, used for generations with few cells
//   NG = 3: 384 threads; the prediction passes of data sets with several parameter segments (up to 170 registers)
//   NG = 4: 512 threads, 1 block per SM; 4x fewer instruction-cache fills per cell (the step's hot code is ~75 kB,
//           over twice the 32 kB L1.5 instruction cache, so every step streams from L2)
// With NG > 1 each group steps behind barriers of its own (ggp_coop_sync), every group runs the block's longest cell, and
// the whole block re-aligns every GGP_COOP_ALIGN_PERIOD steps.
#define GGP_COOP_BLOCK(NG) ((NG) * GGP_COOP_ROLES * 32)
#define GGP_COOP_SEG_SMEM 8   // parameter sets (segments) staged in shared memory by the prediction passes
// dynamic shared memory of the cooperative kernels: [math tables][scratch columns]
#define GGP_COOP_SCRATCH_OFF (sizeof(GgpMathTables))
#define GGP_COOP_SMEM_BYTES(NG) (GGP_COOP_SCRATCH_OFF + (size_t)(NG) * GGP_CS_COUNT * GGP_COOP_CELLS * sizeof(double))
__device__ __forceinline__ void ggp_coop_stage_tables(GgpMathTables* sm) { ggp_stage_tables(sm); }   // ends with a block barrier

// barrier of one 4-warp group (NG > 1: named barrier 1 + group, the groups of a block drift freely) or of the whole block
template <int NG>
__device__ __forceinline__ void ggp_coop_sync(int group) {
    if (NG > 1) asm volatile("bar.sync %0, 128;" ::"r"(group + 1) : "memory");
    else __syncthreads();
}

// 8-byte asynchronous copy global -> shared (no register holds the value while it is in flight)
__device__ __forceinline__ void ggp_cp_async8(double* smem_dst, const double* gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void ggp_cp_async_wait() { asm volatile("cp.async.wait_all;" ::: "memory"); }

constexpr int GGP_COOP_ALIGN_PERIOD = 4;   // steps between the block-wide re-alignments of the groups (NG > 1)

// Profiling aid (never in the shipped build): -DGGP_PHASE_CLOCKS accumulates, per role, the SM clocks spent inside each
// phase and waiting at each barrier of the likelihood step (ggp_debug_phase_clocks reads them; tools/phase_clocks.py).
#ifdef GGP_PHASE_CLOCKS
__device__ unsigned long long ggp_phase_clk[GGP_COOP_ROLES][10];
// per-warp accumulators in shared memory, flushed once per block (contended global atomics inside the loop would show up
// in role 0's cp.async wait)
#define GGP_CLK_DECL                                                      \
    __shared__ unsigned long long s_clk[32][10];                          \
    if (lane < 10) s_clk[warp][lane] = 0;                                 \
    __syncwarp();                                                         \
    long long clk_last = clock64();
#define GGP_CLK_MARK(slot)                                                \
    if (!PRED && lane == 0) {                                             \
        volatile unsigned long long* q = &s_clk[warp][slot];              \
        const unsigned long long acc = *q;   /* a memory operation first: BAR.SYNC.DEFER_BLOCKING lets the clock read run ahead of the barrier */ \
        const long long now = clock64();                                  \
        *q = acc + (unsigned long long)(now - clk_last);                  \
        clk_last = now;                                                   \
    }
#define GGP_CLK_FLUSH                                                     \
    __syncwarp();                                                         \
    if (!PRED && lane < 10) atomicAdd(&ggp_phase_clk[role][lane], s_clk[warp][lane]);
#else
#define GGP_CLK_DECL
#define GGP_CLK_MARK(slot)
#define GGP_CLK_FLUSH
#endif

// PRED = false: likelihood (likelihood.h:36-103, one parameter vector per blockIdx.y); PRED = true: prediction_forward
// (predictions.h:93-150): parameters by segment, the posterior of every point stored to A.out_fwd.
// UNI (PRED only): the data set has one segment, so the parameters are block-uniform like the likelihood's (no per-lane
// parameter pointers, no segment look-ups: the registers those cost are what keeps the prediction passes at 3 groups)
template <int NG, bool PRED = false, bool UNI = false>
__global__ void __launch_bounds__(GGP_COOP_BLOCK(NG), NG == 1 ? 3 : (NG <= 4 ? 4 / NG : 1)) ggp_loglik_coop_kernel(const GgpDevForest F, const GgpFwdArgs A) {
    constexpr bool SEGS = PRED && !UNI;   // per-point parameter sets
    GgpMathTables& T = *reinterpret_cast<GgpMathTables*>(ggp_smem);
    __shared__ double sp[GGP_NP * (PRED ? GGP_COOP_SEG_SMEM : 1)];   // LIK: the vector's parameters; PRED: the first parameter sets
    __shared__ int s_steps[NG * GGP_COOP_ROLES];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int group = warp / GGP_COOP_ROLES, role = warp & (GGP_COOP_ROLES - 1);
    const int v = PRED ? 0 : blockIdx.y;
    if (!PRED && threadIdx.x < GGP_NP)
        sp[threadIdx.x] = A.params ? A.params[(int64_t)(A.v0 + v) * GGP_NP + threadIdx.x] : A.inline_params[(A.v0 + v) * GGP_NP + threadIdx.x];
    if (PRED && (int)threadIdx.x < GGP_NP * min(A.n_seg, GGP_COOP_SEG_SMEM)) sp[threadIdx.x] = A.params[threadIdx.x];
    // parameters of segment s: from shared memory when staged (a per-step pointer chase through global memory otherwise)
    const bool seg_staged = A.n_seg <= GGP_COOP_SEG_SMEM;
    auto seg_params = [&](int s) -> const double* { return seg_staged ? sp + GGP_NP * s : A.params + GGP_NP * s; };
    ggp_coop_stage_tables(&T);   // ends with a block barrier
    GgpScratch S;
    S.base = reinterpret_cast<double*>(ggp_smem + GGP_COOP_SCRATCH_OFF) + (size_t)group * GGP_CS_COUNT * GGP_COOP_CELLS + lane;
    S.stride = GGP_COOP_CELLS;

    const int gidx = blockIdx.x * NG + group;                  // 32-cell group inside this generation
    const int in_gen = gidx * GGP_COOP_CELLS + lane;
    const bool active = in_gen < A.n_slots;
    const int slot = A.slot0 + (active ? in_gen : 0);
    int64_t off = 0;
    int n = 0, parent = -1;
    if (active) {
        off = F.s_off[slot];
        n = F.s_n[slot];
        parent = F.s_parent[slot];
    }
    const int64_t vstride = (int64_t)A.v_count * F.n_cells, vbase = (int64_t)v * F.n_cells;
    const int seg0 = (SEGS && active) ? F.seg[off] : 0;
    double own = 0.0;
    int t = 0;
    int64_t from = off;
    __syncthreads();   // sp
    const double* p = SEGS ? seg_params(seg0) : sp;
    if (active) {
        if (parent < 0) {
            if (role == 0) {   // root: first update on the full matrix
                double mu[4], C[16];
                ggp_root_start(mu, C, nullptr, F, p, off, &T, [&](double ll) {
                    own = own + ll;
                    if (!PRED && ll != ll) GGP_NAN_MIN(A.nan_key + A.v0 + v, F.s_dfs0[slot]);
                });
                if (PRED) ggp_store20(A.out_fwd + 20 * off, mu, C);
                GgpState s;
                ggp_state_from16(s, mu, C);
#pragma unroll
                for (int k = 0; k < 4; ++k) S[GGP_CS_ST + k] = s.m[k];
#pragma unroll
                for (int k = 0; k < 10; ++k) S[GGP_CS_ST + 4 + k] = s.c[k];
            }
        } else {   // daughter: mother's last posterior; the division gap is step "-1"
            for (int k = role; k < 14; k += GGP_COOP_ROLES) S[GGP_CS_ST + k] = A.state[k * vstride + vbase + parent];
            t = -1;
            from = F.s_off[parent] + F.s_n[parent] - 1;
        }
    }
    const int steps = active ? n - 1 - t : 0;
    int max_steps = __reduce_max_sync(0xffffffffu, steps);   // same value in the group's four warps (same 32 cells)
    if (NG > 1) {   // every group runs the block's longest cell
        if (lane == 0) s_steps[warp] = max_steps;
        __syncthreads();
#pragma unroll
        for (int i = 0; i < NG * GGP_COOP_ROLES; ++i) max_steps = max(max_steps, s_steps[i]);
    }
    const GgpOuParams ou_lik = ggp_ou(sp, false);   // LIK: one parameter vector for the whole block
    // pow(gamma_lambda, 3) depends on the parameters only: once per thread (LIK) / per staged segment (PRED), not per step
    __shared__ double s_gl3[GGP_COOP_SEG_SMEM];
    if (PRED && seg_staged && (int)threadIdx.x < A.n_seg) s_gl3[threadIdx.x] = ggp_pow(sp[GGP_NP * threadIdx.x + 1], 3.0, &T);
    if (PRED) __syncthreads();
    const double gl3_lik = (!PRED && role == 3) ? ggp_pow(sp[1], 3.0, &T) : GGP_NO_GL3;
    int prev_seg = -1;   // PRED: segment of the previous step's parameters (the elementary exponentials are reused if unchanged)
    // The measurements of a step (t_to, t_from, x, g) sit in scratch slots GGP_CS_IN + 4 * (step & 1); role 0 fetches
    // those of the NEXT step with cp.async while the current step computes (the loads retire behind a whole step
    // of arithmetic and occupy no registers).
    if (role == 0 && steps > 0) {
        const int64_t at = off + t + 1;
        S[GGP_CS_IN + 0] = F.time[at];
        S[GGP_CS_IN + 1] = F.time[from];
        S[GGP_CS_IN + 2] = F.x[at];
        S[GGP_CS_IN + 3] = F.g[at];
    }
    // PRED: segment of the point a step leaves from / arrives at; the next step's is fetched one step ahead
    int seg_from = (SEGS && active) ? F.seg[from] : 0;
    int seg_at = (SEGS && steps > 0) ? F.seg[off + t + 1] : 0;
    ggp_coop_sync<NG>(group);
    bool pend = false;   // LIK, role 0: a log-evidence term is pending in GGP_CS_LL
    GGP_CLK_DECL
    for (int it = 0; it < max_steps; ++it) {
        const bool live = it < steps;
        const int in = GGP_CS_IN + 4 * (it & 1);
        // re-align the block's groups every GGP_COOP_ALIGN_PERIOD steps (instruction-cache sharing: the groups then fetch the same code at about the same time)
        if (NG > 1 && it % GGP_COOP_ALIGN_PERIOD == 0) __syncthreads();
        GGP_CLK_MARK(0)
        const int seg_next = (SEGS && it + 1 < steps) ? F.seg[off + t + 2] : 0;
        if (role == 0 && it + 1 < steps) {
            const int64_t at = off + t + 2;
            const int nx = GGP_CS_IN + 4 * ((it + 1) & 1);
            ggp_cp_async8(&S[nx + 0], F.time + at);
            ggp_cp_async8(&S[nx + 1], F.time + at - 1);
            ggp_cp_async8(&S[nx + 2], F.x + at);
            ggp_cp_async8(&S[nx + 3], F.g + at);
        }
        const double* pt = p;   // parameters of the point the step arrives at
        if (SEGS && live) {
            p = seg_params(seg_from);
            pt = seg_params(seg_at);
        }
        if (live) {
            const double dt = S[in + 0] - S[in + 1];
            // same dt (and parameters) as this cell's previous step: GGP_CS_GE still holds the elementary exponentials
            const bool ge_same = role == 0 && it > 0 && dt == S[GGP_CS_K + GGP_K_T] && (!SEGS || seg_from == prev_seg);
            // LIK: the previous step's log-evidence term, left pending by phase 3, is finished inside role 0's phase 0 (ggp_coop.cuh)
            const bool take_ll = !PRED && role == 0 && pend;
            double ll = 0.0;
            ggp_coop_run_phase(0, role, S, SEGS ? ggp_ou(p, false) : ou_lik, dt, &T, ge_same, GGP_NO_GL3, take_ll ? &ll : nullptr);
            if (take_ll) {
                own = own + ll;
                if (ll != ll) GGP_NAN_MIN(A.nan_key + A.v0 + v, F.s_dfs0[slot] + t);
                pend = false;
            }
            prev_seg = seg_from;
        }
        GGP_CLK_MARK(1)
        ggp_coop_sync<NG>(group);
        GGP_CLK_MARK(2)
#pragma unroll
        for (int ph = 1; ph < GGP_COOP_PHASES; ++ph) {
            if (live) ggp_coop_run_phase(ph, role, S, SEGS ? ggp_ou(p, false) : ou_lik, 0.0, &T, false,
                                         PRED ? (seg_staged ? s_gl3[seg_from] : GGP_NO_GL3) : gl3_lik);
            GGP_CLK_MARK(1 + 2 * ph)
            ggp_coop_sync<NG>(group);
            GGP_CLK_MARK(2 + 2 * ph)
        }
        if (live) {
            const double ll = PRED ? ggp_coop_ph3_pred<false>(role, S, t < 0, p, pt, S[in + 2], S[in + 3], F.model, &T, A.out_fwd + 20 * (off + t + 1))
                                   : ggp_coop_ph3<true>(role, S, t < 0, p, S[in + 2], S[in + 3], F.model, &T);
            (void)ll;
            ++t;
            from = off + t;
            seg_from = seg_at;
            seg_at = seg_next;
            if (!PRED && role == 0) pend = true;
        }
        if (role == 0) ggp_cp_async_wait();
        GGP_CLK_MARK(7)
        ggp_coop_sync<NG>(group);
        GGP_CLK_MARK(8)
    }
    GGP_CLK_FLUSH
    if (!PRED && role == 0 && pend) {   // the last point's term
        const double ll = ggp_coop_ll_deferred(GGP_SLOTS_REF(S), &T);
        own = own + ll;
        if (ll != ll) GGP_NAN_MIN(A.nan_key + A.v0 + v, F.s_dfs0[slot] + t);
    }
    if (active && (F.s_d1[slot] >= 0 || F.s_d2[slot] >= 0)) {
        for (int k = role; k < 14; k += GGP_COOP_ROLES) A.state[k * vstride + vbase + slot] = S[GGP_CS_ST + k];
    }
    if (!PRED && role == 0) {
        if (active && A.cell_ll) A.cell_ll[(int64_t)(A.v0 + v) * F.n_cells + F.s_cell[slot]] = own;
        double bs = own;   // fixed-order reduction over the block's 32 cells
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) bs = bs + __shfl_xor_sync(0xffffffffu, bs, o);
        if (lane == 0 && gidx * GGP_COOP_CELLS < A.n_slots) A.partial[(int64_t)v * A.n_partial + A.partial0 + gidx] = bs;
    }
}

// ------------------------------------------------------------------------------------------------
// prediction_backward (predictions.h:368-444), cells processed from the leaves upward, one launch per generation.
// Role 0 builds the cell's starting belief (ggp_cell.cuh: ggp_leaf_start, ggp_mother_start); the time-reversed steps then
// run through the same four phases as the forward passes with the sign-flipped parameters (mean_cov_model_r, :191-198).
// ------------------------------------------------------------------------------------------------
template <int NG, bool UNI = false>
__global__ void __launch_bounds__(GGP_COOP_BLOCK(NG), NG == 1 ? 3 : (NG <= 4 ? 4 / NG : 1)) ggp_backward_coop_kernel(const GgpDevForest F, const GgpBwdArgs A) {
    GgpMathTables& T = *reinterpret_cast<GgpMathTables*>(ggp_smem);
    __shared__ int s_steps[NG * GGP_COOP_ROLES];
    __shared__ double sp[GGP_NP * GGP_COOP_SEG_SMEM];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int group = warp / GGP_COOP_ROLES, role = warp & (GGP_COOP_ROLES - 1);
    if ((int)threadIdx.x < GGP_NP * min(A.n_seg, GGP_COOP_SEG_SMEM)) sp[threadIdx.x] = A.params[threadIdx.x];
    const bool seg_staged = A.n_seg <= GGP_COOP_SEG_SMEM;
    auto seg_params = [&](int s) -> const double* { return seg_staged ? sp + GGP_NP * s : A.params + GGP_NP * s; };
    ggp_coop_stage_tables(&T);
    GgpScratch S;
    S.base = reinterpret_cast<double*>(ggp_smem + GGP_COOP_SCRATCH_OFF) + (size_t)group * GGP_CS_COUNT * GGP_COOP_CELLS + lane;
    S.stride = GGP_COOP_CELLS;

    const int gidx = blockIdx.x * NG + group;
    const int in_gen = gidx * GGP_COOP_CELLS + lane;
    const bool active = in_gen < A.n_slots;
    const int slot = A.slot0 + (active ? in_gen : 0);
    int64_t off = 0, from = 0;
    int n = 0, t = 0;
    if (active) {
        off = F.s_off[slot];
        n = F.s_n[slot];
        const int d1 = F.s_d1[slot], d2 = F.s_d2[slot];
        const bool leaf = d1 < 0 && d2 < 0;
        const int da = d1 >= 0 ? d1 : d2;
        t = leaf ? n - 1 : n;                       // mothers start at a virtual point: the daughters' first time
        from = leaf ? off + t : F.s_off[da];
        if (role == 0) {
            const double* p0 = UNI ? A.params : A.params + GGP_NP * F.seg[off + n - 1];
            double mu[4], C[16];
            GgpState s;
            if (leaf) {
                ggp_leaf_start(mu, C, F, A.fwd, A.bwd, p0, from);
                ggp_state_from16(s, mu, C);
                if (t == 0) ggp_store20(A.bstate + 20 * (int64_t)slot, mu, C);   // one-point leaf: no step follows
            } else {
                ggp_mother_start(mu, C, A.bstate, d1, d2, p0, F.model);
                ggp_state_from16(s, mu, C);
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) S[GGP_CS_ST + k] = s.m[k];
#pragma unroll
            for (int k = 0; k < 10; ++k) S[GGP_CS_ST + 4 + k] = s.c[k];
        }
    }
    const int steps = active ? t : 0;
    int max_steps = __reduce_max_sync(0xffffffffu, steps);
    if (NG > 1) {
        if (lane == 0) s_steps[warp] = max_steps;
        __syncthreads();
#pragma unroll
        for (int i = 0; i < NG * GGP_COOP_ROLES; ++i) max_steps = max(max_steps, s_steps[i]);
    }
    if (role == 0 && steps > 0) {
        const int64_t at = off + t - 1;
        S[GGP_CS_IN + 0] = F.time[from];
        S[GGP_CS_IN + 1] = F.time[at];
        S[GGP_CS_IN + 2] = F.x[at];
        S[GGP_CS_IN + 3] = F.g[at];
    }
    int seg_at = (!UNI && steps > 0) ? F.seg[off + t - 1] : 0;
    const GgpOuParams ou_uni = ggp_ou(sp, true);   // UNI: one (sign-flipped) parameter set for the whole block
    ggp_coop_sync<NG>(group);
    for (int it = 0; it < max_steps; ++it) {
        const bool live = it < steps;
        const int in = GGP_CS_IN + 4 * (it & 1);
        if (NG > 1 && it % GGP_COOP_ALIGN_PERIOD == 0) __syncthreads();
        const int64_t at = off + t - 1;   // the point this step arrives at
        const int seg_next = (!UNI && it + 1 < steps) ? F.seg[at - 1] : 0;
        if (role == 0 && it + 1 < steps) {
            const int nx = GGP_CS_IN + 4 * ((it + 1) & 1);
            ggp_cp_async8(&S[nx + 0], F.time + at);
            ggp_cp_async8(&S[nx + 1], F.time + at - 1);
            ggp_cp_async8(&S[nx + 2], F.x + at - 1);
            ggp_cp_async8(&S[nx + 3], F.g + at - 1);
        }
        const double* pp = A.params;
        if (live) {
            pp = UNI ? sp : seg_params(seg_at);
            const double dt = S[in + 0] - S[in + 1];
            ggp_coop_run_phase(0, role, S, UNI ? ou_uni : ggp_ou(pp, true), dt, &T);
        }
        ggp_coop_sync<NG>(group);
#pragma unroll
        for (int ph = 1; ph < GGP_COOP_PHASES; ++ph) {
            if (live) ggp_coop_run_phase(ph, role, S, UNI ? ou_uni : ggp_ou(pp, true), 0.0, &T);
            ggp_coop_sync<NG>(group);
        }
        if (live) {
            ggp_coop_store_reversed(role, S, A.bwd + 20 * at);
            --t;
            ggp_coop_ph3_pred<false>(role, S, false, pp, pp, S[in + 2], S[in + 3], F.model, &T,
                                     t == 0 ? A.bstate + 20 * (int64_t)slot : nullptr);
            seg_at = seg_next;
        }
        if (role == 0) ggp_cp_async_wait();
        ggp_coop_sync<NG>(group);
    }
}

// ------------------------------------------------------------------------------------------------
// Carry mode (SURVEY.md H3): the reference's roots keep their covariance object across evaluations; only its
// diagonal is reset (predictions.h:64-78), so evaluation v of a root starts from the off-diagonals evaluation v-1
// left at the root's last point.  The vectors of a batch therefore form a sequential chain per root: this kernel runs
// the roots' generation for ALL vectors of the chunk one after the other (32 roots per block, four roles), the other
// generations use ggp_loglik_coop_kernel with one block column per vector.  A.carry [n_roots][16] in/out.
// ------------------------------------------------------------------------------------------------
#define GGP_COOP_SMEM_BYTES_CHAIN (GGP_COOP_SCRATCH_OFF + (size_t)GGP_CS_COUNT_CHAIN * GGP_COOP_CELLS * sizeof(double))

__global__ void __launch_bounds__(GGP_COOP_BLOCK(1), 3) ggp_loglik_chain_coop_kernel(const GgpDevForest F, const GgpFwdArgs A) {
    GgpMathTables& T = *reinterpret_cast<GgpMathTables*>(ggp_smem);
    __shared__ double sp[GGP_NP];
    const int role = threadIdx.x >> 5, lane = threadIdx.x & 31;
    ggp_coop_stage_tables(&T);
    GgpScratch S;
    S.base = reinterpret_cast<double*>(ggp_smem + GGP_COOP_SCRATCH_OFF) + lane;
    S.stride = GGP_COOP_CELLS;
    const GgpScratch carry{&S[GGP_CS_CARRY + 4], S.stride};
    const int in_gen = blockIdx.x * GGP_COOP_CELLS + lane;
    const bool active = in_gen < A.n_slots;
    const int slot = A.slot0 + (active ? in_gen : 0);
    int64_t off = 0;
    int n = 0;
    if (active) {
        off = F.s_off[slot];
        n = F.s_n[slot];
        for (int i = role; i < 16; i += GGP_COOP_ROLES) carry[i] = A.carry[16 * (int64_t)F.s_root[slot] + i];
    }
    const int steps = active ? n - 1 : 0;
    const int max_steps = __reduce_max_sync(0xffffffffu, steps);
    const int64_t vstride = (int64_t)A.v_count * F.n_cells;
    for (int v = 0; v < A.v_count; ++v) {
        __syncthreads();
        if (threadIdx.x < GGP_NP) sp[threadIdx.x] = A.params[(int64_t)(A.v0 + v) * GGP_NP + threadIdx.x];
        __syncthreads();
        const double* p = sp;
        const int64_t vbase = (int64_t)v * F.n_cells;
        double own = 0.0;
        if (active && role == 0) {   // first update on the full matrix with the stale off-diagonals
            double mu[4], C[16];
            ggp_root_start(mu, C, &carry, F, p, off, &T, [&](double ll) {
                own = own + ll;
                if (ll != ll) GGP_NAN_MIN(A.nan_key + A.v0 + v, F.s_dfs0[slot]);
            });
#pragma unroll
            for (int i = 0; i < 16; ++i) carry[i] = C[i];
            GgpState s;
            ggp_state_from16(s, mu, C);
#pragma unroll
            for (int k = 0; k < 4; ++k) S[GGP_CS_ST + k] = s.m[k];
#pragma unroll
            for (int k = 0; k < 10; ++k) S[GGP_CS_ST + 4 + k] = s.c[k];
            if (steps > 0) {
                S[GGP_CS_IN + 0] = F.time[off + 1];
                S[GGP_CS_IN + 1] = F.time[off];
                S[GGP_CS_IN + 2] = F.x[off + 1];
                S[GGP_CS_IN + 3] = F.g[off + 1];
            }
        }
        __syncthreads();
        const GgpOuParams ou = ggp_ou(p, false);
        for (int it = 0; it < max_steps; ++it) {
            const bool live = it < steps;
            const int in = GGP_CS_IN + 4 * (it & 1);
            if (role == 0 && it + 1 < steps) {
                const int64_t at = off + it + 2;
                const int nx = GGP_CS_IN + 4 * ((it + 1) & 1);
                ggp_cp_async8(&S[nx + 0], F.time + at);
                ggp_cp_async8(&S[nx + 1], F.time + at - 1);
                ggp_cp_async8(&S[nx + 2], F.x + at);
                ggp_cp_async8(&S[nx + 3], F.g + at);
            }
            if (live) ggp_coop_run_phase(0, role, S, ou, S[in + 0] - S[in + 1], &T);
            __syncthreads();
#pragma unroll
            for (int ph = 1; ph < GGP_COOP_PHASES; ++ph) {
                if (live) ggp_coop_run_phase(ph, role, S, ou, 0.0, &T);
                __syncthreads();
            }
            if (live) {
                const bool last = it + 1 == steps;   // the complete posterior of the last point is what the next vector inherits
                const double ll = ggp_coop_ph3_out<true>(role, S, false, p, p, S[in + 2], S[in + 3], F.model, &T,
                                                         GgpOutScratch{S, last ? (int)GGP_CS_CARRY : -1});
                if (role == 0) {
                    own = own + ll;
                    if (ll != ll) GGP_NAN_MIN(A.nan_key + A.v0 + v, F.s_dfs0[slot] + it + 1);
                }
            }
            if (role == 0) ggp_cp_async_wait();
            __syncthreads();
        }
        if (active && (F.s_d1[slot] >= 0 || F.s_d2[slot] >= 0)) {
            for (int k = role; k < 14; k += GGP_COOP_ROLES) A.state[k * vstride + vbase + slot] = S[GGP_CS_ST + k];
        }
        if (role == 0) {
            if (active && A.cell_ll) A.cell_ll[(int64_t)(A.v0 + v) * F.n_cells + F.s_cell[slot]] = own;
            double bs = own;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) bs = bs + __shfl_xor_sync(0xffffffffu, bs, o);
            if (lane == 0) A.partial[(int64_t)v * A.n_partial + A.partial0 + blockIdx.x] = bs;
        }
    }
    __syncthreads();
    if (active) {
        for (int i = role; i < 16; i += GGP_COOP_ROLES) A.carry[16 * (int64_t)F.s_root[slot] + i] = carry[i];
    }
}

// ---- self-test of the fast paths the cooperative step adds on top of the strict math (ggp_math_eval fn 5, 6) ----
// one warp per block, lane = test case, a full scratch column per lane (the slot helpers assume the 32-cell stride)
//   fn 5: x = pow base, y = exp argument -> out[5 i] = pow(x, 1.5 + i % 3), out[5 i + 1..4] = exp of y, y / 2, -y, y + 1
//         through ggp_pow_exp_slots (main paths interleaved, anything else through the out-of-line routines)
//   fn 6: x[5 i ..] = quadratic form, S00, S01, S10, S11 -> the log-evidence term as role 0's phase 0 finishes it
//         (shared-reciprocal division and log's main path inline, ggp_coop_ll_deferred otherwise)
__global__ void __launch_bounds__(GGP_COOP_CELLS) ggp_coop_math_kernel(int fn, int64_t n, const double* __restrict__ x,
                                                                      const double* __restrict__ y, double* __restrict__ out) {
    GgpMathTables& T = *reinterpret_cast<GgpMathTables*>(ggp_smem);
    ggp_coop_stage_tables(&T);
    GgpScratch S;
    S.base = reinterpret_cast<double*>(ggp_smem + GGP_COOP_SCRATCH_OFF) + threadIdx.x;
    S.stride = GGP_COOP_CELLS;
    const int64_t i = (int64_t)blockIdx.x * GGP_COOP_CELLS + threadIdx.x;
    if (i >= n) return;
    if (fn == 5) {
        S[GGP_CS_EC + 0] = y[i]; S[GGP_CS_EC + 1] = y[i] / 2; S[GGP_CS_EC + 2] = -y[i]; S[GGP_CS_EC + 3] = y[i] + 1;
        out[5 * i] = ggp_pow_exp_slots(x[i], 1.5 + (double)(i % 3), GGP_SLOTS_REF(S), GGP_CS_EC, 4, &T);
        for (int k = 0; k < 4; ++k) out[5 * i + 1 + k] = S[GGP_CS_EC + k];
    } else {
        for (int k = 0; k < 14; ++k) S[GGP_CS_ST + k] = k < 4 ? 1.0 : (k == 4 || k == 8 || k == 11 || k == 13 ? 1.0 : 0.125);
        for (int k = 0; k < 5; ++k) S[GGP_CS_LL + k] = x[5 * i + k];
        GgpOuParams p;
        p.ml = 0.01; p.gl = 0.01; p.sl2 = 1e-5; p.mq = 10.; p.gq = 0.01; p.sq2 = 0.1; p.b = 1e-3;
        double ll = 0.0;
        ggp_coop_run_phase(0, 0, S, p, 1.0, &T, false, GGP_NO_GL3, &ll);
        out[i] = ll;
    }
}
