// C ABI of the engine (include/ttrnn_b200.h): validation, planning, workspace layout and
// the host-side launch sequence (layer by layer, time chunk by time chunk).
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "tt_kernels.cuh"
#include "tt_proj.cuh"
#include "tt_cell.cuh"
#include "tt_gemm.cuh"
#include "tt_tc.cuh"
#include "tt_ge2e.cuh"
#include "tt_dense.cuh"
#include "tt_bidir.cuh"
#include "tt_dropout.cuh"
#include "tt_static.cuh"
#include "tt_static_api.h"

namespace {

thread_local std::string g_err = "";
std::atomic<long long> g_launches{0};
std::atomic<long long> g_tc_launches{0};      // launches of the tcgen05 GEMMs (tt_tc.cuh) among them
std::atomic<long long> g_opt_rows{0};
std::atomic<long long> g_opt_chunk{0};
std::atomic<long long> g_opt_chunk_bytes{4LL << 30};
std::atomic<long long> g_opt_static{1};
std::atomic<long long> g_opt_srows_fwd{0}, g_opt_srows_bwd{0};
// budget for keeping only the hh pre-activations u (G*H floats per row and step) so that backward skips the
// final stage of the chain recompute (measured on cfg2: see profiles/)
std::atomic<long long> g_opt_save_u_bytes{16LL << 30};
// dense route of the batched ih projection (tt_gemm.cuh): used when I*G*H <= ratio% of the chain's
// multiply-adds per row (and the shape fits the GEMM tiles); 0 disables
std::atomic<long long> g_opt_row_plan{1};      // two-phase row plans of the static BPTT kernels
std::atomic<long long> g_opt_dense_ih{1};
// split backward (cfg5-class chains): accumulate the hh core gradients through the dense order
// dW_hh^T = H_prev^T delta (one GEMM pass, then an H-row projection onto the cores) instead of a second
// chain pass per row (recompute + dX chain + dW chain): 4.2 M vs 3.5 M multiply-adds per row at H = 1024,
// but in GEMM form (measured ~67 % vs ~50 % of the FFMA peak)
// dense-route row GEMMs: 128 x 256 CTA tiles (8 x 16 thread tiles, one CTA per SM) when N % 256 == 0.  Off: measured
// 7 % slower than the 128 x 128 / two-CTA variant on cfg3 and cfg4 (8 warps per SM do not cover the LDS latency).
std::atomic<long long> g_opt_gemm_wide{0};
std::atomic<long long> g_opt_dense_hh{1};
std::atomic<long long> g_opt_split_kept{1};    // kept gates: prefer the dX-only BPTT variants + dense hh core gradients
std::atomic<long long> g_opt_dense_ratio{130};
// dense-route GEMMs on the tensor cores (tt_tc.cuh: tcgen05 3xTF32, TMA-staged) where the shape fits; 0 = FP32 FFMA kernels
std::atomic<long long> g_opt_tc_gemm{1};
// zero-pad TT ranks that are not multiples of 4 so that the static kernels apply (make_eff_desc); 0 = runtime-shape kernels
std::atomic<long long> g_opt_rank_pad{1};
// multi-layer backward: run the weight-gradient work of layer l (dW GEMMs, projections onto the cores, partial folds) on a
// second stream, on the SMs the BPTT kernel of layer l - 1 leaves idle (its grid is rows / rows-per-CTA, e.g. 98 of 148 at
// cfg3).  Needs a second set of the per-layer scratch buffers; single-chunk plans only.  0 = everything on the caller's stream
std::atomic<long long> g_opt_bwd_overlap{1};
// multi-layer stacks: split the batch into two ROW GROUPS that run the whole stack independently on two streams (see
// plan_row_groups).  A layer-pass of one launch leaves SMs idle whenever rows / rows-per-CTA is not a multiple of the SM
// count (cfg3: 128 five-row CTAs forward, 148 + 98 CTAs backward on 148 SMs); with two groups the tail group of layer l
// runs beside the head group of layer l + 1 (forward) / l - 1 (backward).  0 = one group (every launch on the caller's stream),
// 1 = planned, >= 4 = force group 0 to that many rows whatever the plan says (tests)
std::atomic<long long> g_opt_row_groups{1};
// d3 r8 TT-LSTM chains: run static kernels with cores 0 and 1 contracted (tts::Merge01: one stage and 10 % of the
// multiply-adds fewer per step).  1 (default) = the dX-only BPTT kernels only: the forward keeps the three-core chain, so
// outputs, states and everything computed from them stay bit-identical to merge_cores = 0 and only the BPTT sums are
// reordered; 2 = the forward kernels as well (another ~3 % on cfg3, but h_t is rounded differently, which a GE2E loss
// backward amplifies: cfg9 parameter gradients move by ~1e-5 relative); 0 = the three-core chain everywhere.  The fused BPTT
// kernels, the runtime-shape kernels and the gradient-logging path always run the three-core chain.
std::atomic<long long> g_opt_merge_cores{1};

// Snapshot of every option that decides a buffer layout or a kernel route.  ttrnn_rnn_workspace_bytes() takes it from the
// process-wide options and stamps it into ttrnn_rnn_workspace.plan; forward and backward run from THAT copy, so a
// ttrnn_set_option() between a forward and its backward (another model, another thread) cannot change how `saved` and
// the scratch buffers are interpreted.  Helpers read the calling thread's current snapshot `t_opt`.
struct Opts {
    long long rows, chunk, chunk_bytes, stat, srows_fwd, srows_bwd, save_u_bytes, row_plan, dense_ih, gemm_wide,
        dense_hh, split_kept, dense_ratio, tc_gemm, rank_pad, bwd_overlap, row_groups, merge_cores;
};
constexpr int kOptFields = sizeof(Opts) / sizeof(long long);
constexpr long long kPlanMagic = 0x7474726E6E706C36LL;          // "ttrnnpl6"
// plan words: [0] magic, [1 .. kOptFields] options, then the row-group split (group count, rows of group 0), then 1 when
// the state buffers are per layer (TTRNN_WS_LAYER_STATES), then 1 when `saved` keeps the masked layer inputs of the
// dropout entry points (TTRNN_WS_DROPOUT), then 1 when the plan is for the projected entry points (TTRNN_WS_PROJ)
constexpr int kPlanGroups = kOptFields + 1, kPlanRows0 = kOptFields + 2, kPlanLayerStates = kOptFields + 3,
              kPlanDropout = kOptFields + 4, kPlanProj = kOptFields + 5;
static_assert(kOptFields + 6 <= TTRNN_PLAN_WORDS, "plan does not fit ttrnn_rnn_workspace.plan");
thread_local Opts t_opt;
inline int merge_fwd() { return t_opt.merge_cores >= 2 ? 1 : 0; }    // contracted forward variants (merge_cores = 2)
inline int merge_bwd() { return t_opt.merge_cores >= 1 ? 1 : 0; }    // contracted dX-only BPTT variants (merge_cores >= 1)

Opts snapshot_options() {
    Opts o;
    o.rows = g_opt_rows.load(); o.chunk = g_opt_chunk.load(); o.chunk_bytes = g_opt_chunk_bytes.load();
    o.stat = g_opt_static.load(); o.srows_fwd = g_opt_srows_fwd.load(); o.srows_bwd = g_opt_srows_bwd.load();
    o.save_u_bytes = g_opt_save_u_bytes.load(); o.row_plan = g_opt_row_plan.load();
    o.dense_ih = g_opt_dense_ih.load(); o.gemm_wide = g_opt_gemm_wide.load(); o.dense_hh = g_opt_dense_hh.load();
    o.split_kept = g_opt_split_kept.load(); o.dense_ratio = g_opt_dense_ratio.load(); o.tc_gemm = g_opt_tc_gemm.load();
    o.rank_pad = g_opt_rank_pad.load(); o.bwd_overlap = g_opt_bwd_overlap.load(); o.row_groups = g_opt_row_groups.load();
    o.merge_cores = g_opt_merge_cores.load();
    return o;
}
void plan_store(const Opts &o, int64_t *plan) {
    plan[0] = kPlanMagic;
    memcpy(plan + 1, &o, sizeof o);
}
bool plan_load(const int64_t *plan, Opts *o) {
    if (!plan || plan[0] != kPlanMagic) return false;
    memcpy(o, plan + 1, sizeof *o);
    return true;
}

// ---- optional per-kernel event timing (bench only) -----------------------------------------
// R / ctas / rows / steps: rows per CTA, grid size, batch rows and timesteps of a recurrent-kernel launch (0 for the other kinds)
struct TimedLaunch { int kind; cudaEvent_t a, b; int R, ctas; long long rows; int steps; };
struct LaunchRecord { int kind, R, ctas; long long rows; int steps; double ms; };
std::mutex g_time_mu;
std::vector<TimedLaunch> g_timed;
std::vector<LaunchRecord> g_records;           // per-launch durations of the last ttrnn_kernel_times() call
std::atomic<int> g_timing{0};
constexpr size_t kMaxTimed = 8192;

struct KernelTimer {
    cudaEvent_t a = nullptr, b = nullptr;
    int kind;
    cudaStream_t st;
    bool on = false;
    int R, ctas;
    long long rows;
    int steps;
    KernelTimer(int kind_, cudaStream_t st_, int R_ = 0, int ctas_ = 0, long long rows_ = 0, int steps_ = 0)
        : kind(kind_), st(st_), R(R_), ctas(ctas_), rows(rows_), steps(steps_) {
        if (!g_timing.load()) return;
        {
            std::lock_guard<std::mutex> lk(g_time_mu);
            if (g_timed.size() >= kMaxTimed) return;
        }
        if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return;
        on = true;
        cudaEventRecord(a, st);
    }
    ~KernelTimer() {
        if (!on) return;
        cudaEventRecord(b, st);
        std::lock_guard<std::mutex> lk(g_time_mu);
        g_timed.push_back({kind, a, b, R, ctas, rows, steps});
    }
};

int fail(const char *fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return 1;
}

#define CU_CHECK(expr)                                                                       \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) return fail("%s failed: %s", #expr, cudaGetErrorString(_e)); \
    } while (0)

struct DevInfo {
    int sms = 0;
    int smem_optin = 0;
    bool ok = false;
};

int get_dev(DevInfo *d) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess)
        return fail("no CUDA device available (%s): ttrnn_b200 has no CPU path", cudaGetErrorString(e));
    CU_CHECK(cudaDeviceGetAttribute(&d->sms, cudaDevAttrMultiProcessorCount, dev));
    CU_CHECK(cudaDeviceGetAttribute(&d->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    d->ok = true;
    return 0;
}

// Where layer l's initial state, final state and their gradients live.  stride 0 is the reference's contract
// (lstm.py:120-121,135): one (B, H) block seeds every layer, only the last layer's final state comes back and takes an
// upstream gradient, and d_h0 / d_c0 receive the sum over layers.  stride > 0 (TTRNN_WS_LAYER_STATES): every state buffer
// is (L, B, H) and layer l's block starts l * stride floats in.  The stride is the FULL batch's B * H, also inside a row
// group, whose pointers the entry points have already moved to the group's first row.  With a projection the h-state
// blocks are B * P and the c-state blocks B * H: `c` selects the c-state stride.
struct StateMap {
    long long stride = 0, cstride = 0;
    template <class P> P init(P p, int l, bool c = false) const {                                             // h0, c0, d_h0, d_c0
        const long long s = c ? cstride : stride;
        return (p && s) ? p + l * s : p;
    }
    template <class P> P fin(P p, int l, int L, bool c = false) const {                                       // hT, cT, d_hT, d_cT
        if (stride) return p ? p + l * (c ? cstride : stride) : p;
        return l == L - 1 ? p : nullptr;
    }
};

inline int gates_of(int cell) { return cell == TTRNN_CELL_LSTM ? 4 : 3; }
inline long long r4(long long v) { return (v + 3) & ~3LL; }

// ---- tile heuristics --------------------------------------------------------------------
int choose_fwd_tile(const StagePlan &s, int R) {
    if (s.K % 4 != 0 || s.N % 4 != 0) return TT_TILE_GEN;
    const long long per = (long long)R * s.Mrow * s.N / TT_NTHREADS;
    if (s.N % 8 == 0 && per >= 64) return TT_TILE_8x8;
    if (s.N % 8 == 0 && per >= 32) return TT_TILE_4x8;
    if (per >= 32) return TT_TILE_8x4;
    if (per >= 16) return TT_TILE_4x4;
    if (per >= 8) return TT_TILE_2x4;
    return TT_TILE_1x4;
}
int choose_bd_tile(const StagePlan &s, int R) {
    if (s.K % 4 != 0) return TT_TILE_GEN;
    const long long per = (long long)R * s.Mrow * s.K / TT_NTHREADS;
    if (s.K % 8 == 0 && per >= 64) return TT_TILE_8x8;
    if (s.K % 8 == 0 && per >= 32) return TT_TILE_4x8;
    if (per >= 32) return TT_TILE_8x4;
    if (per >= 16) return TT_TILE_4x4;
    if (per >= 8) return TT_TILE_2x4;
    return TT_TILE_1x4;
}
int choose_mg(const StagePlan &s, int R) {
    const int tk = (s.K % 4 == 0) ? 4 : 2;
    const int tn = (s.K % 4 == 0 || s.r % 4 == 0) ? 4 : 2;
    const int items = ((s.K + tk - 1) / tk) * ((s.N + tn - 1) / tn);
    const int M = R * s.Mrow;
    int mg = TT_NTHREADS / items;
    if (mg < 1) mg = 1;
    const int cap = M / 4 > 1 ? M / 4 : 1;
    return mg > cap ? cap : mg;
}
void fill_tiles(const ChainPlan &p, int R, int *tf, int *tb, int *mg) {
    for (int k = 0; k < p.d; ++k) {
        if (tf) tf[k] = choose_fwd_tile(p.st[k], R);
        if (tb) tb[k] = choose_bd_tile(p.st[k], R);
        if (mg) mg[k] = choose_mg(p.st[k], R);
    }
}

// ---- shared-memory footprints (floats) --------------------------------------------------
long long smem_ttlin_fwd(const ChainPlan &p, int R) {
    return p.w_floats + (long long)R * (p.in_BS + p.pp_floats[0] + p.pp_floats[1] + p.g_BS);
}
long long smem_rnn_fwd(const ChainPlan &p, int R, int H, int G) {
    return p.w_floats + (G == 4 ? 0 : r4(G * H)) + r4((long long)R * H) + r4((long long)R * G * H) +
           (long long)R * (p.g_BS + p.in_BS + p.pp_floats[0] + p.pp_floats[1]);
}
// backward footprints split into the part that does not depend on where the X_k slots live ...
long long smem_ttlin_bwd_fixed(const ChainPlan &p, int R) {
    return 2LL * p.w_floats + r4(p.n_out) + (long long)R * (p.g_BS + p.in_BS);
}
long long smem_rnn_bwd_fixed(const ChainPlan &p, int R, int H, int G) {
    return 2LL * p.w_floats + (G == 4 ? 0 : 2 * r4(G * H)) + (long long)R * (p.g_BS + p.in_BS) +
           r4((long long)R * G * H) + 3 * r4((long long)R * H);
}

template <class F>
int pick_rows(F smem_floats, int smem_limit_bytes, int rmax, long long units, int sms, int want_ctas_per_sm) {
    int R = 0;
    for (int r = 1; r <= rmax; ++r)
        if (smem_floats(r) * 4 <= smem_limit_bytes) R = r;
    if (R == 0) return 0;
    const long long opt = t_opt.rows;
    if (opt > 0) return (int)(opt < R ? opt : R);
    while (R > 1 && (units + R - 1) / R < (long long)want_ctas_per_sm * sms) --R;
    return R;
}

// Backward launch configuration: rows per CTA, slot placement (shared vs spill), footprints.
struct BwdCfg {
    ChainPlan p;            // plan with the slot placement applied
    int R = 0;
    size_t smem = 0;        // bytes
    long long spill = 0;    // floats of global spill per CTA
};

template <class Fixed>
int plan_bwd(const ChainPlan &base, Fixed fixed_floats, const DevInfo &dv, long long units, BwdCfg *c,
             const char *what) {
    c->p = base;
    auto total = [&](int r) { return fixed_floats(r) + (long long)r * base.all_floats; };
    int R = pick_rows(total, dv.smem_optin, 8, units, dv.sms, 2);
    if (R > 0) {
        c->R = R;
        c->smem = (size_t)total(R) * 4;
        c->spill = 0;
        return 0;
    }
    // one row per CTA, largest X_k slots moved to the L2-resident spill area
    const long long budget = dv.smem_optin / 4 - fixed_floats(1);
    if (budget < 0)
        return fail("%s: cores alone need %lld bytes of shared memory (limit %d): unsupported TT shape", what,
                    fixed_floats(1) * 4, dv.smem_optin);
    tt_place_slots(&c->p, budget);
    c->R = 1;
    c->smem = (size_t)(fixed_floats(1) + c->p.all_floats) * 4;
    c->spill = c->p.spill_floats;
    return 0;
}

// projected LSTM: footprints of k_rnn_fwd_proj / k_rnn_bwd_proj (tt_proj.cuh), hh chain p and projection chain q
long long smem_rnn_fwd_proj(const ChainPlan &p, const ChainPlan &q, int R, int H) {
    const long long pp0 = p.pp_floats[0] > q.pp_floats[0] ? p.pp_floats[0] : q.pp_floats[0];
    const long long pp1 = p.pp_floats[1] > q.pp_floats[1] ? p.pp_floats[1] : q.pp_floats[1];
    return p.w_floats + q.w_floats + r4((long long)R * H) + r4((long long)R * 4 * H) +
           (long long)R * (p.g_BS + p.in_BS + q.in_BS + q.g_BS + pp0 + pp1);
}
long long smem_rnn_bwd_proj_fixed(const ChainPlan &p, const ChainPlan &q, int R, int H, int P) {
    return 2LL * (p.w_floats + q.w_floats) + (long long)R * (p.g_BS + q.g_BS + p.in_BS) + r4((long long)R * 4 * H) +
           r4((long long)R * P) + 2 * r4((long long)R * H);
}
struct BwdProjCfg {
    ChainPlan p, q;         // plans with the slot placement applied
    int R = 0;
    size_t smem = 0;        // bytes
    long long spill = 0;    // floats of global spill per CTA (both chains)
};
// plan_bwd for the two chains of k_rnn_bwd_proj: when their kept X_k slots do not fit one row per CTA, the projection
// chain's largest slots move to the spill area first, then the hh chain's
int plan_bwd_proj(const ChainPlan &p, const ChainPlan &q, int H, int P, const DevInfo &dv, long long units, BwdProjCfg *c) {
    c->p = p;
    c->q = q;
    auto fixed = [&](int r) { return smem_rnn_bwd_proj_fixed(p, q, r, H, P); };
    auto total = [&](int r) { return fixed(r) + (long long)r * (p.all_floats + q.all_floats); };
    int R = pick_rows(total, dv.smem_optin, 8, units, dv.sms, 2);
    if (R > 0) {
        c->R = R;
        c->smem = (size_t)total(R) * 4;
        c->spill = 0;
        return 0;
    }
    const long long budget = dv.smem_optin / 4 - fixed(1);
    if (budget < 0)
        return fail("projected hh backward: cores alone need %lld bytes of shared memory (limit %d): unsupported TT shape",
                    fixed(1) * 4, dv.smem_optin);
    if (budget >= p.all_floats) {
        tt_place_slots(&c->q, budget - p.all_floats);
    } else {
        tt_place_slots(&c->q, 0);
        tt_place_slots(&c->p, budget);
    }
    c->R = 1;
    c->smem = (size_t)(fixed(1) + c->p.all_floats + c->q.all_floats) * 4;
    c->spill = c->p.spill_floats + c->q.spill_floats;
    return 0;
}

template <class K>
int grid_for(K kernel, size_t smem_bytes, long long ntiles, const DevInfo &dv, int *grid) {
    CU_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
    int occ = 0;
    CU_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, TT_NTHREADS, smem_bytes));
    if (occ < 1) return fail("kernel does not fit on an SM (%zu bytes of shared memory)", smem_bytes);
    if (occ > 4) occ = 4;
    long long g = (long long)occ * dv.sms;
    if (g > ntiles) g = ntiles;
    *grid = (int)g;
    return 0;
}
constexpr int kMaxSlotsPerSM = 4;

// ---- descriptor validation / parameter blob layout -----------------------------------------
struct LayerPlan {
    ChainPlan ih, hh;
    ChainPlan hr;                                                     // projection W_hr (H -> P), when P > 0
    long long off_ih_cores, off_ih_bias, off_hh_cores, off_hh_bias;   // floats into the blob
    long long off_hr_cores;
};
struct RnnPlan {
    int G = 0;
    int P = 0;               // projection size (TTRNN_WS_PROJ); 0 = none, the layer output is H wide
    long long param_floats = 0;
    LayerPlan layer[TTRNN_MAX_LAYERS];
    int out_width(const ttrnn_rnn_desc *d) const { return P ? P : d->hidden_size; }
};

// pj: the projection of the _proj entry points, or nullptr
int build_rnn_plan(const ttrnn_rnn_desc *d, RnnPlan *rp, const ttrnn_rnn_proj *pj = nullptr) {
    if (!d) return fail("null descriptor");
    if (d->cell != TTRNN_CELL_LSTM && d->cell != TTRNN_CELL_GRU) return fail("unknown cell kind %d", d->cell);
    if (d->num_layers < 1 || d->num_layers > TTRNN_MAX_LAYERS)
        return fail("num_layers %d out of range [1, %d]", d->num_layers, TTRNN_MAX_LAYERS);
    if (d->input_size < 1 || d->hidden_size < 1) return fail("input_size / hidden_size must be positive");
    if (d->batch < 1 || d->seq_len < 1) return fail("batch and seq_len must be >= 1 (got %lld, %d)", (long long)d->batch, d->seq_len);
    rp->G = gates_of(d->cell);
    rp->P = 0;
    if (pj) {
        if (d->cell != TTRNN_CELL_LSTM) return fail("a projection (proj_size) needs an LSTM descriptor");
        if (pj->proj_size < 1 || pj->proj_size >= d->hidden_size)
            return fail("proj_size %d out of range [1, hidden_size %d)", pj->proj_size, d->hidden_size);
        rp->P = pj->proj_size;
    }
    const int GH = rp->G * d->hidden_size, W = rp->out_width(d);
    long long off = 0;
    for (int l = 0; l < d->num_layers; ++l) {
        LayerPlan &lp = rp->layer[l];
        int rc = tt_build_plan(&d->ih[l], &lp.ih);
        if (rc) return fail("layer %d: malformed ih TT shape (code %d)", l, rc);
        rc = tt_build_plan(&d->hh[l], &lp.hh);
        if (rc) return fail("layer %d: malformed hh TT shape (code %d)", l, rc);
        const int want_in = (l == 0) ? d->input_size : W;
        if (lp.ih.n_in != want_in || lp.ih.n_out != GH)
            return fail("layer %d: ih TT matrix is %d x %d, expected %d x %d", l, lp.ih.n_out, lp.ih.n_in, GH, want_in);
        if (lp.hh.n_in != W || lp.hh.n_out != GH)
            return fail("layer %d: hh TT matrix is %d x %d, expected %d x %d", l, lp.hh.n_out, lp.hh.n_in, GH, W);
        lp.off_ih_cores = off; off += lp.ih.core_floats;
        lp.off_ih_bias = off;  if (d->has_bias) off += GH;
        lp.off_hh_cores = off; off += lp.hh.core_floats;
        lp.off_hh_bias = off;  if (d->has_bias) off += GH;
        lp.off_hr_cores = off;
        if (rp->P) {
            rc = tt_build_plan(&pj->hr[l], &lp.hr);
            if (rc) return fail("layer %d: malformed hr TT shape (code %d)", l, rc);
            if (lp.hr.n_in != d->hidden_size || lp.hr.n_out != rp->P)
                return fail("layer %d: hr TT matrix is %d x %d, expected %d x %d", l, lp.hr.n_out, lp.hr.n_in, rp->P,
                            d->hidden_size);
            off += lp.hr.core_floats;
        }
    }
    rp->param_floats = off;
    return 0;
}

// ---- kernel routes of a recurrent layer -------------------------------------------------------------------------
// Every caller that needs to know which recurrent kernel a layer runs (workspace layout, row-group planner, describe,
// the launch paths) asks these functions, so that the plan they report and model is the one that launches.

// input mode of layer l: a single input feature (I = 1) is folded into the recurrent kernel as a rank-one term
inline int layer_mode(const ttrnn_rnn_desc *d, int l) {
    return (l == 0 && d->input_size == 1) ? tts::MODE_RANK1 : tts::MODE_XG;
}

// statically specialised forward kernel of layer l at B rows on `sms` SMs, or nullptr (runtime-shape kernel).  A projected
// layer has none: its chains run on the runtime-shape kernels k_rnn_fwd_proj / k_rnn_bwd_proj.
const TtsRnnFwdEntry *fwd_route(const ttrnn_rnn_desc *d, const RnnPlan &rp, int l, long long B, int sms) {
    if (!t_opt.stat || rp.P) return nullptr;
    return tts_find_rnn_fwd(&d->hh[l], d->cell, layer_mode(d, l), B, sms, (int)t_opt.srows_fwd, merge_fwd());
}

// ---- rank padding -----------------------------------------------------------------------------------------------
// The statically specialised kernels need inner TT ranks that are multiples of 4 (tt_static.cuh).  A chain whose ranks
// are not (the reference's own GE2E default is n_cores = 2, rank = 2: encoder/params_model.py:15-16) is mathematically
// identical to the chain with every inner rank rounded up and the cores zero-padded along their rank axes.  When ALL
// hh chains of the padded stack have a registered static kernel, the call runs on the padded descriptor: the parameter
// blob is expanded into scratch by k_pad_cores, and the backward cuts the real gradient block out of the padded one.
// The padded chain executes more multiply-adds (r = 2 -> 4: 2x on the rank-bound stages), but on kernels that are
// 5-10x faster than the runtime-shape fallback.
constexpr int kMaxPadEntries = TTRNN_MAX_LAYERS * 2 * (TTRNN_MAX_CORES + 1);
struct PadEntry { int src, dst, r, mid, rn, rnp; };       // core (r, mid, rn) at src -> (rp, mid, rnp) at dst (floats)
struct PadTable { int n; PadEntry e[kMaxPadEntries]; };

__global__ void __launch_bounds__(256) k_pad_cores(const __grid_constant__ PadTable t, const float *__restrict__ src,
                                                   float *__restrict__ dst) {
    const PadEntry en = t.e[blockIdx.x];
    // iterate over the SOURCE extents; the added rank slices are zeroed by the memset the host issues before this kernel
    const int n = en.r * en.mid * en.rn;
    for (int i = threadIdx.x; i < n; i += 256) {
        const int b = i % en.rn, m = (i / en.rn) % en.mid, a = i / (en.rn * en.mid);
        dst[en.dst + (a * en.mid + m) * en.rnp + b] = src[en.src + i];
    }
}
__global__ void __launch_bounds__(256) k_unpad_cores(const __grid_constant__ PadTable t, const float *__restrict__ padded,
                                                     float *__restrict__ real) {
    const PadEntry en = t.e[blockIdx.x];
    const int n = en.r * en.mid * en.rn;
    for (int i = threadIdx.x; i < n; i += 256) {
        const int b = i % en.rn, m = (i / en.rn) % en.mid, a = i / (en.rn * en.mid);
        real[en.src + i] = padded[en.dst + (a * en.mid + m) * en.rnp + b];
    }
}

struct EffDesc {
    ttrnn_rnn_desc d;          // descriptor the kernels run on (padded ranks when `padded`)
    bool proj = false;         // + the projection `pj` (TTRNN_WS_PROJ)
    ttrnn_rnn_proj pj;
    bool padded = false;
    PadTable tab;
    long long pad_floats = 0;  // floats of the padded parameter blob
};

// pj: a projected stack is never padded (no static kernel would take it)
int make_eff_desc(const ttrnn_rnn_desc *d, const ttrnn_rnn_proj *pj, const DevInfo *dv, EffDesc *e) {
    e->d = *d;
    e->padded = false;
    e->pad_floats = 0;
    e->tab.n = 0;
    e->proj = pj != nullptr;
    if (pj) e->pj = *pj;
    if (!t_opt.stat || !t_opt.rank_pad || !dv || pj) return 0;
    RnnPlan real;
    if (build_rnn_plan(d, &real)) return 1;
    bool any = false;
    ttrnn_rnn_desc p = *d;
    for (int l = 0; l < d->num_layers; ++l)
        for (int side = 0; side < 2; ++side) {
            ttrnn_tt_shape &sh = side ? p.hh[l] : p.ih[l];
            for (int k = 1; k < sh.d; ++k) {
                const int rp = (sh.ranks[k] + 3) & ~3;
                if (rp != sh.ranks[k]) { sh.ranks[k] = rp; any = true; }
            }
        }
    if (!any) return 0;
    for (int l = 0; l < d->num_layers; ++l)
        if (!fwd_route(&p, real, l, d->batch, dv->sms)) return 0;     // padding would not reach a static kernel
    RnnPlan pad;
    if (build_rnn_plan(&p, &pad)) return 0;
    const int GH = real.G * d->hidden_size;
    PadTable &t = e->tab;
    for (int l = 0; l < d->num_layers; ++l)
        for (int side = 0; side < 2; ++side) {
            const ttrnn_tt_shape &sr = side ? d->hh[l] : d->ih[l], &sp = side ? p.hh[l] : p.ih[l];
            long long so = side ? real.layer[l].off_hh_cores : real.layer[l].off_ih_cores;
            long long po = side ? pad.layer[l].off_hh_cores : pad.layer[l].off_ih_cores;
            for (int k = 0; k < sr.d; ++k) {
                PadEntry en;
                en.src = (int)so; en.dst = (int)po;
                en.r = sr.ranks[k]; en.mid = sr.out_modes[k] * sr.in_modes[k]; en.rn = sr.ranks[k + 1]; en.rnp = sp.ranks[k + 1];
                t.e[t.n++] = en;
                so += (long long)sr.ranks[k] * en.mid * sr.ranks[k + 1];
                po += (long long)sp.ranks[k] * en.mid * sp.ranks[k + 1];
            }
            if (d->has_bias) {
                PadEntry en;
                en.src = (int)(side ? real.layer[l].off_hh_bias : real.layer[l].off_ih_bias);
                en.dst = (int)(side ? pad.layer[l].off_hh_bias : pad.layer[l].off_ih_bias);
                en.r = 1; en.mid = GH; en.rn = 1; en.rnp = 1;
                t.e[t.n++] = en;
            }
        }
    e->d = p;
    e->padded = true;
    e->pad_floats = r4(pad.param_floats);
    return 0;
}

// ---- dense route of the batched ih projection (tt_gemm.cuh) -------------------------------------
constexpr int kDenseMaxSplit = 40;

long long chain_macs(const ChainPlan &p) {
    long long m = 0;
    for (int k = 0; k < p.d; ++k) m += (long long)p.st[k].Mrow * p.st[k].K * p.st[k].N;
    return m;
}
// forward / recompute / dW^T all need: G*H % 128 == 0, I % 4 == 0
// `shape` (optional): when no statically specialised chain kernel is registered for it, the alternative to the
// dense order is the ~5-10x slower runtime-shape kernel, so the dense order is allowed up to 4x the chain's MACs
bool dense_ih_ok(const ChainPlan &ih, const ttrnn_tt_shape *shape = nullptr) {
    if (!t_opt.dense_ih) return false;
    if (ih.n_out % ttg::BN != 0 || ih.n_in % 4 != 0 || ih.n_in < 4 || ih.n_in > 2048) return false;
    long long ratio = t_opt.dense_ratio;
    if (shape && !(t_opt.stat && tts_find_ttl_fwd(shape, 1 << 20)) && ratio < 400) ratio = 400;
    return (long long)ih.n_in * ih.n_out * 100 <= chain_macs(ih) * ratio;
}
// dX = delta * W additionally needs I % 128 == 0
bool dense_ih_bwd_ok(const ChainPlan &ih, bool want_dx, const ttrnn_tt_shape *shape = nullptr) {
    return dense_ih_ok(ih, shape) && (!want_dx || ih.n_in % ttg::BN == 0);
}

bool dense_hh_dw_ok(const ChainPlan &hh) {
    return t_opt.dense_hh && hh.n_out % ttg::BN == 0 && hh.n_in % 4 == 0 && hh.n_in <= 2048;
}

// Static BPTT route of layer l at B rows on `sms` SMs.  `mode` is an argument because a rank-one layer 0 whose input
// gradient is requested runs the MODE_XG kernels.  `kept`: the forward kept this layer's gate activations (the kept-gates
// kernels are then preferred where registered); Tc: timesteps per chunk of the layout.
struct BwdRoute {
    int nph = 0;                                       // phases of the row plan; 0 = runtime-shape kernel
    const TtsRnnBwdEntry *e[2] = {nullptr, nullptr};   // kernel of each phase
    long long row0[2] = {0, 0}, rows[2] = {0, 0};      // first row and row count of each phase
    bool kept = false;       // the kernels consume the kept gate activations
    bool split = false;      // dX-only kernels: the hh core gradients are computed outside the recurrent kernel ...
    bool dense_hh = false;   // ... by the dense accumulation dW_hh^T = H_prev^T delta (else a second chain pass)
    bool split_r1 = false;   // split behind a rank-one input: bias / W_ih-column gradients stay in the kernel's slots
};

int bwd_route(const ttrnn_rnn_desc *d, const RnnPlan &rp, int l, int mode, long long B, int sms, bool kept, long long Tc,
              BwdRoute *r) {
    *r = BwdRoute();
    if (!t_opt.stat || rp.P) return 0;
    const ttrnn_tt_shape *hh = &d->hh[l];
    const int srows = (int)t_opt.srows_bwd;
    const TtsRnnBwdEntry *be = tts_find_rnn_bwd(hh, d->cell, mode, B, sms, srows, 0, 0, merge_bwd());
    if (kept) {
        // the dX-only ("split") variants need the dense accumulation of the hh core gradients; with a rank-one input the
        // delta buffer must also hold the whole sequence (single-chunk plans)
        const bool split_ok = dense_hh_dw_ok(rp.layer[l].hh) && t_opt.split_kept && (mode != tts::MODE_RANK1 || Tc >= d->seq_len);
        if (const TtsRnnBwdEntry *bs = tts_find_rnn_bwd(hh, d->cell, mode, B, sms, srows, 2, split_ok, merge_bwd())) be = bs;
    }
    if (!be) return 0;
    r->nph = 1;
    r->e[0] = be;
    r->rows[0] = B;
    // row plan: one phase, or two when a tail variant beats a mostly idle last wave
    if ((!be->split || be->saved == 2) && t_opt.row_plan) {
        const TtsRnnBwdEntry *pe[2];
        long long pr0[2], pr[2];
        const int np = tts_plan_rnn_bwd(hh, d->cell, mode, B, sms, srows, be->saved, be->split && be->saved == 2, merge_bwd(),
                                        pe, pr0, pr);
        if (np >= 1) {
            r->nph = np;
            for (int q = 0; q < np; ++q) { r->e[q] = pe[q]; r->row0[q] = pr0[q]; r->rows[q] = pr[q]; }
        }
    }
    r->kept = r->e[0]->saved == 2;
    r->split = r->e[0]->split != 0;
    r->dense_hh = r->split && dense_hh_dw_ok(rp.layer[l].hh);
    r->split_r1 = r->split && mode == tts::MODE_RANK1;
    // split variants behind a projected input take the hh bias gradient from the ih side (LSTM only); the rank-one
    // variants keep every bias / W_ih-column gradient in the kernel's own slot and work for both cells
    if (r->split && d->cell != TTRNN_CELL_LSTM && !r->split_r1)
        return fail("internal: split BPTT variants with a projected input compute the hh bias gradient from the ih side "
                    "(LSTM only); %s is registered for a GRU", r->e[0]->name);
    if (r->split_r1 && !r->dense_hh)
        return fail("internal: rank-one split BPTT variant %s selected without the dense hh core-gradient route", r->e[0]->name);
    return 0;
}

struct DenseIh {
    float *eye, *wt, *w, *w_hi, *w_lo, *wt_hi, *wt_lo, *dwt, *dbias, *part, *pbias;
};
// forward: identity, W^T (I x G*H), W (G*H x I) and its TF32 hi / lo split (tensor-core route)
long long dense_fwd_floats(const ChainPlan &ih) { return r4((long long)ih.n_in * ih.n_in) + 4 * r4((long long)ih.n_in * ih.n_out); }
// backward adds: hi / lo split of W^T (dX on the tensor cores), dW^T, dbias and the split partials
long long dense_bwd_floats(const ChainPlan &ih) {
    const long long wn = r4((long long)ih.n_in * ih.n_out);
    return dense_fwd_floats(ih) + 3 * wn + r4(ih.n_out) + kDenseMaxSplit * (wn + r4(ih.n_out));
}
// ---- workspace layout --------------------------------------------------------------------
struct RnnLayout {
    int Tc = 0;                 // timesteps per chunk
    long long BTH = 0, BH = 0;
    long long BTW = 0, BW = 0;  // the same for a layer's output width W: P with a projection (h_t, its gradients), else H
    long long xg_floats = 0;
    // saved (floats)
    long long sv_hs = 0, sv_cs = 0, sv_total = 0;
    // fwd scratch (floats)
    long long f_xg = 0, f_sh = 0, f_sc = 0, f_hs = 0, f_aux = 0, f_dense = 0, f_total = 0;
    // bwd scratch (floats)
    long long b_xg = 0, b_dhs = 0, b_sdh = 0, b_sdc = 0, b_part_hh = 0, b_part_ih = 0, b_spill = 0, b_aux = 0, b_dense = 0, b_dense_hh = 0, b_total = 0;
    long long part_stride = 0;  // floats per partial slot
    int nslots = 0;
    // backward overlap: the per-layer buffers (everything from b_xg on) exist twice, set (l & 1) at + set * set_stride
    int overlap = 0;
    long long set_stride = 0;
    // kept gate activations (static kernels, within the save_u_bytes budget): per layer flag and offset into `saved`
    bool kept[TTRNN_MAX_LAYERS] = {};
    long long sv_u[TTRNN_MAX_LAYERS] = {};
    // inter-layer dropout (TTRNN_WS_DROPOUT, L > 1): masked inputs of layers 1 .. L-1 at the end of `saved` (training),
    // one (B, T, H) block at the end of the forward scratch (inference)
    bool masked = false;
    long long sv_drop = 0, f_drop = 0;
};

int build_layout(const ttrnn_rnn_desc *d, const RnnPlan &rp, const DevInfo &dv, RnnLayout *lo, bool keep_masked) {
    const long long B = d->batch, T = d->seq_len, H = d->hidden_size, L = d->num_layers;
    const long long GH = (long long)rp.G * H, W = rp.out_width(d);
    lo->BTH = B * T * H;
    lo->BH = B * H;
    lo->BTW = B * T * W;
    lo->BW = B * W;
    long long tc = t_opt.chunk;
    if (tc <= 0) {
        tc = t_opt.chunk_bytes / (B * GH * 4);
        if (tc < 1) tc = 1;
    }
    if (tc > T) tc = T;
    lo->Tc = (int)tc;
    lo->xg_floats = r4(B * tc * GH);
    const bool lstm = d->cell == TTRNN_CELL_LSTM;
    // saved: inner-layer outputs, then cell states of every layer
    lo->sv_hs = 0;
    lo->sv_cs = r4((L - 1) * lo->BTW);
    lo->sv_total = lo->sv_cs + (lstm ? r4(L * lo->BTH) : 0);
    // kept gate activations of the static recurrent kernels ("save_u_bytes" budget, default 16 GiB): 4*H floats per row
    // and step (LSTM i,f,g,o; GRU r,z,n,u_n) -- backward skips the final stage of the recompute and all gate math.  Every
    // layer whose forward and kept-gates backward are static keeps them, or none does.  The dense accumulation of the hh
    // core gradients is sized for a split backward with or without kept gates.
    bool can_keep[TTRNN_MAX_LAYERS] = {};
    long long kept_floats = 0, dhh = 0;
    if (t_opt.stat)
        for (int l = 0; l < L; ++l) {
            BwdRoute recompute, keep;
            if (bwd_route(d, rp, l, layer_mode(d, l), B, dv.sms, false, tc, &recompute) ||
                bwd_route(d, rp, l, layer_mode(d, l), B, dv.sms, true, tc, &keep))
                return 1;
            can_keep[l] = keep.kept && fwd_route(d, rp, l, B, dv.sms);
            if (can_keep[l]) kept_floats += r4(B * T * 4 * H);
            if ((recompute.dense_hh || keep.dense_hh) && dense_bwd_floats(rp.layer[l].hh) > dhh)
                dhh = dense_bwd_floats(rp.layer[l].hh);
        }
    const bool keep_all = kept_floats > 0 && kept_floats * 4 <= t_opt.save_u_bytes;
    for (int l = 0; l < L; ++l) {
        lo->kept[l] = keep_all && can_keep[l];
        if (lo->kept[l]) { lo->sv_u[l] = lo->sv_total; lo->sv_total += r4(B * T * 4 * H); }
    }
    lo->masked = keep_masked && L > 1;
    if (lo->masked) { lo->sv_drop = lo->sv_total; lo->sv_total += r4((L - 1) * lo->BTW); }
    // forward scratch
    long long o = 0;
    lo->f_xg = o; o += lo->xg_floats;
    lo->f_sh = o; o += r4(lo->BW);
    lo->f_sc = o; o += r4(lo->BH);
    lo->f_hs = o; o += (L > 1 ? 2 * r4(lo->BTW) : 0);     // used only when nothing is saved
    lo->f_aux = o; o += r4(GH) + 4;                       // rank-one input mode: dense W_ih column + a 1.0f
    long long dfw = 0, dbw = 0;                           // dense ih route: identity, W^T (+ W, dW^T, split partials)
    for (int l = 0; l < L; ++l)
        if (dense_ih_ok(rp.layer[l].ih, &d->ih[l])) {
            if (dense_fwd_floats(rp.layer[l].ih) > dfw) dfw = dense_fwd_floats(rp.layer[l].ih);
            if (dense_bwd_floats(rp.layer[l].ih) > dbw) dbw = dense_bwd_floats(rp.layer[l].ih);
        }
    lo->f_dense = o; o += dfw;
    lo->f_drop = o; o += lo->masked ? r4(lo->BTW) : 0;
    lo->f_total = o;
    // backward scratch
    long long maxp = 0;
    for (int l = 0; l < L; ++l) {
        long long a = rp.layer[l].ih.core_floats + GH, b = rp.layer[l].hh.core_floats + 3 * GH;
        if (rp.P) b += rp.layer[l].hr.core_floats;
        if (a > maxp) maxp = a;
        if (b > maxp) maxp = b;
    }
    lo->part_stride = r4(maxp);
    lo->nslots = dv.sms * kMaxSlotsPerSM;
    o = 0;
    lo->b_dhs = o; o += (L > 1 ? 2 * r4(lo->BTW) : 0);
    lo->b_sdh = o; o += r4(lo->BW);
    lo->b_sdc = o; o += r4(lo->BH);
    const long long set_base = o;                         // per-layer buffers from here on
    lo->b_xg = o; o += lo->xg_floats;
    lo->b_part_hh = o; o += lo->part_stride * lo->nslots;
    lo->b_part_ih = o; o += lo->part_stride * lo->nslots;
    // spill area for backward X_k slots that do not fit in shared memory (worst layer, either kernel)
    long long spill = 0;
    for (int l = 0; l < L; ++l) {
        BwdCfg c;
        const ChainPlan &hh = rp.layer[l].hh, &ih = rp.layer[l].ih;
        const int Hh = (int)H, Gg = rp.G;
        if (rp.P) {
            BwdProjCfg cq;
            if (plan_bwd_proj(hh, rp.layer[l].hr, Hh, rp.P, dv, B, &cq)) return 1;
            if (cq.spill > spill) spill = cq.spill;
        } else {
            if (plan_bwd(hh, [&](int r) { return smem_rnn_bwd_fixed(hh, r, Hh, Gg); }, dv, B, &c, "hh backward")) return 1;
            if (c.spill > spill) spill = c.spill;
        }
        if (plan_bwd(ih, [&](int r) { return smem_ttlin_bwd_fixed(ih, r); }, dv, B * tc, &c, "ih backward")) return 1;
        if (c.spill > spill) spill = c.spill;
    }
    lo->b_spill = o; o += r4(spill) * lo->nslots;
    lo->b_aux = o; o += 2 * r4(GH) + 4;                   // rank-one input mode: W_ih column, its gradient, a 1.0f
    lo->b_dense = o; o += dbw;
    lo->b_dense_hh = o; o += dhh;                         // split backward: dense accumulation of the hh core gradients
    lo->overlap = (t_opt.bwd_overlap && t_opt.stat && L > 1 && tc == T) ? 1 : 0;
    if (lo->overlap) {
        lo->set_stride = r4(o - set_base);
        o = set_base + 2 * lo->set_stride;
    }
    lo->b_total = o;
    return 0;
}

// Everything a call derives from its descriptor: the effective (possibly rank-padded) descriptor, its parameter plan and
// its workspace layout on the device `dv`.
struct CallPlan {
    DevInfo dv;
    EffDesc eff;
    RnnPlan rp;         // of eff.d
    RnnLayout lo;
    const ttrnn_rnn_desc *d() const { return &eff.d; }
    const ttrnn_rnn_proj *pj() const { return eff.proj ? &eff.pj : nullptr; }
};

// keep_masked: the plan carries TTRNN_WS_DROPOUT; pj: the projection of the _proj entry points (TTRNN_WS_PROJ) or nullptr.
// The effective descriptor carries the projection from here on.
int plan_call(const ttrnn_rnn_desc *d_in, const DevInfo &dv, CallPlan *cp, bool keep_masked = false,
              const ttrnn_rnn_proj *pj = nullptr) {
    cp->dv = dv;
    if (build_rnn_plan(d_in, &cp->rp, pj) || make_eff_desc(d_in, pj, &dv, &cp->eff)) return 1;
    if (cp->eff.padded && build_rnn_plan(&cp->eff.d, &cp->rp)) return 1;
    return build_layout(&cp->eff.d, cp->rp, dv, &cp->lo, keep_masked);
}

// ---- inter-layer dropout (tt_dropout.cuh) --------------------------------------------------------------------------
// the mask of one call: nullptr = no dropout; row0 = global batch row of the row group's first row
struct DropCall {
    float p;
    uint64_t seed, offset;
    long long row0;
};
static ttdrop::Mask drop_mask(const DropCall &dc, long long row0, int boundary) {
    ttdrop::Mask m;
    m.seed = dc.seed; m.offset = dc.offset; m.row0 = row0; m.boundary = (unsigned)boundary;
    const double keep = 1.0 - (double)dc.p;
    m.thr = (unsigned long long)(keep * 4294967296.0);
    m.scale = keep > 0.0 ? (float)(1.0 / keep) : 0.f;
    return m;
}
static bool aligned16(const void *p) { return ((uintptr_t)p & 15) == 0; }
// y = (x + rev(xr)) * mask / (1 - p) over (B, T, F), rows from row0; yr (optional) receives y reversed in time
static int launch_dropout(const DevInfo &dv, long long B, int T, int F, const DropCall &dc, long long row0, int boundary,
                          const float *x, const float *xr, float *y, float *yr, cudaStream_t st) {
    const ttdrop::Mask m = drop_mask(dc, row0, boundary);
    if (F % 4 == 0 && aligned16(x) && aligned16(xr) && aligned16(y) && aligned16(yr)) {
        const long long n = B * (long long)T * (F / 4);
        ttdrop::k_dropout_4<<<ttdrop::grid_for(n, dv.sms), ttdrop::NT, 0, st>>>(x, xr, y, yr, n, T, F / 4, m);
    } else {
        const long long n = B * (long long)T * F;
        ttdrop::k_dropout_1<<<ttdrop::grid_for(n, dv.sms), ttdrop::NT, 0, st>>>(x, xr, y, yr, n, T, F, m);
    }
    ++g_launches;
    CU_CHECK(cudaGetLastError());
    return 0;
}

// ---- launch helpers ------------------------------------------------------------------------
int launch_ttlinear_fwd(const ChainPlan &p, const DevInfo &dv, long long rows, int rows_per_b, const float *x,
                        long long x_bstride, const float *cores, const float *bias, const float *bias2, float *y,
                        long long y_bstride, cudaStream_t st, const ttrnn_tt_shape *shape = nullptr) {
    if (shape && t_opt.stat) {
        if (const TtsTtlFwdEntry *e = tts_find_ttl_fwd(shape, rows)) {
            int occ = 0;
            int rc = e->prepare(&occ);
            if (rc || occ < 1) return fail("static kernel %s cannot be configured (cuda error %d)", e->name, rc);
            long long g = (long long)occ * dv.sms;
            const long long tiles = (rows + e->R - 1) / e->R;
            if (g > tiles) g = tiles;
            tts::TtlFwdSArgs sa;
            memset(&sa, 0, sizeof sa);
            sa.rows = rows; sa.rows_per_b = rows_per_b; sa.x_bstride = x_bstride; sa.y_bstride = y_bstride;
            sa.x = x; sa.cores = cores; sa.bias = bias; sa.bias2 = bias2; sa.y = y;
            {
                KernelTimer tm(TTRNN_K_TTLINEAR_FWD, st);
                rc = e->launch(&sa, (int)g, st);
            }
            ++g_launches;
            if (rc) return fail("static kernel %s launch failed: %s", e->name, cudaGetErrorString((cudaError_t)rc));
            return 0;
        }
    }
    TTLinFwdArgs a;
    memset(&a, 0, sizeof a);
    a.p = p;
    const int R = pick_rows([&](int r) { return smem_ttlin_fwd(p, r); }, dv.smem_optin, 8, rows, dv.sms, 2);
    if (R == 0)
        return fail("TT shape needs %lld bytes of shared memory per row tile (limit %d): unsupported",
                    smem_ttlin_fwd(p, 1) * 4, dv.smem_optin);
    a.R = R;
    fill_tiles(p, R, a.tile, nullptr, nullptr);
    a.rows = rows; a.rows_per_b = rows_per_b; a.x_bstride = x_bstride; a.y_bstride = y_bstride;
    a.x = x; a.cores = cores; a.bias = bias; a.bias2 = bias2; a.y = y;
    const size_t smem = (size_t)smem_ttlin_fwd(p, R) * 4;
    int grid = 0;
    if (grid_for(k_ttlinear_fwd, smem, (rows + R - 1) / R, dv, &grid)) return 1;
    {
        KernelTimer tm(TTRNN_K_TTLINEAR_FWD, st);
        k_ttlinear_fwd<<<grid, TT_NTHREADS, smem, st>>>(a);
    }
    ++g_launches;
    CU_CHECK(cudaGetLastError());
    return 0;
}

int launch_ttlinear_bwd(const ChainPlan &p0, const DevInfo &dv, long long rows, int rows_per_b, const float *x,
                        long long x_bstride, const float *cores, const float *dy, long long dy_bstride, float *dx,
                        long long dx_bstride, float *partial, int nslots, float *spill, int want_dbias,
                        cudaStream_t st, int *slots_used, const ttrnn_tt_shape *shape = nullptr) {
    if (shape && t_opt.stat) {
        if (const TtsTtlBwdEntry *e = tts_find_ttl_bwd(shape, rows, dx != nullptr)) {
            int occ = 0;
            int rc = e->prepare(&occ);
            if (rc || occ < 1) return fail("static kernel %s cannot be configured (cuda error %d)", e->name, rc);
            long long g = (long long)occ * dv.sms;
            const long long tiles = (rows + e->R - 1) / e->R;
            if (g > tiles) g = tiles;
            if (g > nslots) g = nslots;
            tts::TtlBwdSArgs sa;
            memset(&sa, 0, sizeof sa);
            sa.rows = rows; sa.rows_per_b = rows_per_b;
            sa.x_bstride = x_bstride; sa.dy_bstride = dy_bstride; sa.dx_bstride = dx_bstride;
            sa.x = x; sa.cores = cores; sa.dy = dy; sa.dx = dx; sa.partial = partial; sa.want_dbias = want_dbias;
            {
                KernelTimer tm(TTRNN_K_TTLINEAR_BWD, st);
                rc = e->launch(&sa, (int)g, st);
            }
            ++g_launches;
            if (rc) return fail("static kernel %s launch failed: %s", e->name, cudaGetErrorString((cudaError_t)rc));
            if (slots_used && (int)g > *slots_used) *slots_used = (int)g;
            return 0;
        }
    }
    BwdCfg c;
    if (plan_bwd(p0, [&](int r) { return smem_ttlin_bwd_fixed(p0, r); }, dv, rows, &c, "TT matvec backward")) return 1;
    TTLinBwdArgs a;
    memset(&a, 0, sizeof a);
    a.p = c.p;
    a.R = c.R;
    fill_tiles(c.p, c.R, a.tile, a.tile_bd, a.mg);
    a.rows = rows; a.rows_per_b = rows_per_b;
    a.x_bstride = x_bstride; a.dy_bstride = dy_bstride; a.dx_bstride = dx_bstride;
    a.x = x; a.cores = cores; a.dy = dy; a.dx = dx; a.partial = partial; a.want_dbias = want_dbias;
    if (c.spill > 0 && !spill) return fail("internal: spill area required but not provided");
    a.spill = c.spill > 0 ? spill : nullptr;
    int grid = 0;
    if (grid_for(k_ttlinear_bwd, c.smem, (rows + c.R - 1) / c.R, dv, &grid)) return 1;
    if (grid > nslots) grid = nslots;
    {
        KernelTimer tm(TTRNN_K_TTLINEAR_BWD, st);
        k_ttlinear_bwd<<<grid, TT_NTHREADS, c.smem, st>>>(a);
    }
    ++g_launches;
    CU_CHECK(cudaGetLastError());
    if (slots_used && grid > *slots_used) *slots_used = grid;
    return 0;
}

int reduce_partials(const float *partial, int nslots, long long slot_stride, long long off, int n, float *out,
                    cudaStream_t st) {
    if (n <= 0) return 0;
    k_reduce_partials<<<(n + 255) / 256, 256, 0, st>>>(partial + off, nslots, n, slot_stride, out);
    ++g_launches;
    CU_CHECK(cudaGetLastError());
    return 0;
}

int axpy1(const float *src, float *dst, long long n, int accumulate, cudaStream_t st) {
    k_axpy1<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(src, dst, n, accumulate);
    ++g_launches;
    CU_CHECK(cudaGetLastError());
    return 0;
}

// ---- dense route: launch helpers ----------------------------------------------------------------
void dense_carve(float *base, const ChainPlan &ih, bool bwd, DenseIh *D) {
    const long long wn = r4((long long)ih.n_in * ih.n_out);
    D->eye = base; base += r4((long long)ih.n_in * ih.n_in);
    D->wt = base; base += wn;
    D->w = base; base += wn;
    D->w_hi = base; base += wn;
    D->w_lo = base; base += wn;
    D->wt_hi = D->wt_lo = D->dwt = D->dbias = D->part = D->pbias = nullptr;
    if (!bwd) return;
    D->wt_hi = base; base += wn;
    D->wt_lo = base; base += wn;
    D->dwt = base; base += wn;
    D->dbias = base; base += r4(ih.n_out);
    D->part = base; base += kDenseMaxSplit * wn;
    D->pbias = base;
}

// tensor-core route limits: the main TMEM accumulator of k_tc_rows chains K / 8 truncating adds (tt_tc.cuh)
constexpr int kTcMaxKFwd = 512, kTcMaxKGrad = 2048;
bool tc_rows_use(long long rows, int K, int N, bool grad) {
    return t_opt.tc_gemm && ttc::tc_rows_ok(rows, K, N) && K <= (grad ? kTcMaxKGrad : kTcMaxKFwd);
}

int split_tf32(const float *src, float *hi, float *lo, long long n, cudaStream_t st) {
    long long blocks = (n / 4 + 255) / 256;
    if (blocks > 1184) blocks = 1184;
    ttc::k_split_tf32<<<(unsigned)blocks, 256, 0, st>>>(src, hi, lo, n / 4);
    ++g_launches;
    CU_CHECK(cudaGetLastError());
    return 0;
}

// W^T (I x G*H): the TT matvec applied to the rows of the identity; optionally W (G*H x I) as well, and the TF32 hi / lo
// splits the tensor-core GEMMs take as their weight operand (W for the forward projection, W^T for dX)
int dense_prepare(const ChainPlan &ih, const ttrnn_tt_shape *shape, const DevInfo &dv, const float *cores, DenseIh &D,
                  bool need_w, bool split_w, bool split_wt, cudaStream_t st) {
    const int I = ih.n_in, GH = ih.n_out;
    ttg::k_eye<<<(I * I + 255) / 256 > 1024 ? 1024 : (I * I + 255) / 256, 256, 0, st>>>(D.eye, I);
    ++g_launches;
    CU_CHECK(cudaGetLastError());
    if (launch_ttlinear_fwd(ih, dv, I, I, D.eye, 0, cores, nullptr, nullptr, D.wt, 0, st, shape)) return 1;
    if (need_w || split_w) {
        dim3 grid((GH + 31) / 32, (I + 31) / 32);
        ttg::k_transpose<<<grid, 256, 0, st>>>(D.wt, D.w, I, GH);
        ++g_launches;
        CU_CHECK(cudaGetLastError());
    }
    const long long wn = r4((long long)I * GH);
    if (split_w && split_tf32(D.w, D.w_hi, D.w_lo, wn, st)) return 1;
    if (split_wt && split_tf32(D.wt, D.wt_hi, D.wt_lo, wn, st)) return 1;
    return 0;
}

// C[r, :] = A[r, :] * B (+ bias + bias2) over ragged rows (time-chunk views)
int dense_rows_gemm(int kind, const DevInfo &dv, long long rows, int rpb, const float *a, long long a_bstride, int K,
                    const float *b, const float *bt_hi, const float *bt_lo, int N, const float *bias, const float *bias2,
                    float *c, long long c_bstride, bool grad, cudaStream_t st) {
    if (rows < 1 || rows > 0x7fffffffLL) return fail("dense ih projection: row count out of range");
    if (bt_hi && bt_lo && tc_rows_use(rows, K, N, grad)) {
        // tensor cores: tcgen05 3xTF32, Bt (N x K) pre-split into hi / lo
        int rc;
        {
            KernelTimer tm(kind, st);
            rc = ttc::launch_tc_rows(rows, rpb, a, a_bstride, K, bt_hi, bt_lo, N, bias, bias2, c, c_bstride, dv.sms, st, grad);
        }
        if (rc == 0) { ++g_launches; ++g_tc_launches; return 0; }
        if (rc > 0) return fail("k_tc_rows launch failed (code %d)", rc);
        // rc < 0: the views cannot be described by a tensor map (alignment): FP32 FFMA kernel below
    }
    ttg::GemmRowsArgs g;
    memset(&g, 0, sizeof g);
    g.rows = (unsigned)rows; g.K = K; g.N = N;
    g.a.p = a; g.a.bstride = a_bstride; g.a.rpb = rpb; g.a.ld = K;
    g.b = b; g.ldb = N; g.bias = bias; g.bias2 = bias2;
    g.c.p = c; g.c.bstride = c_bstride; g.c.rpb = rpb; g.c.ld = N;
    const bool wide = t_opt.gemm_wide && N % 256 == 0;       // 128 x 256 CTA tile, 8 x 16 thread tile
    const long long tiles = ((rows + 127) / 128) * (N / (wide ? 256 : ttg::BN));
    if (tiles > 0x7fffffffLL) return fail("dense ih projection: too many tiles");
    {
        KernelTimer tm(kind, st);
        if (wide) ttg::k_gemm_rows<8, 4><<<(unsigned)tiles, ttg::NT, 0, st>>>(g);
        else ttg::k_gemm_rows<8, 2><<<(unsigned)tiles, ttg::NT, 0, st>>>(g);
    }
    ++g_launches;
    CU_CHECK(cudaGetLastError());
    return 0;
}

// dwt (I x G*H) (+)= X^T delta over the rows of one chunk; dbias (G*H) (+)= column sums of delta
int dense_dw(const DevInfo &dv, long long rows, int rpb, const float *x, long long x_bstride, int I, const float *delta,
             long long d_bstride, int GH, DenseIh &D, bool accumulate, bool want_bias, cudaStream_t st) {
    if (rows < 1 || rows > 0x7fffffffLL) return fail("dense ih backward: row count out of range");
    if (t_opt.tc_gemm && ttc::tc_red_ok(rows, I, GH)) {
        // tensor cores: tcgen05 3xTF32 with the TMEM accumulator promoted into FP32 registers every 32 k-blocks
        int ns = 0, rc;
        {
            KernelTimer tm(TTRNN_K_GEMM_DW, st);
            rc = ttc::launch_tc_red(rows, rpb, x, x_bstride, I, delta, d_bstride, GH, D.part, want_bias ? D.pbias : nullptr,
                                    dv.sms, kDenseMaxSplit, &ns, st);
        }
        if (rc > 0) return fail("k_tc_red launch failed (code %d)", rc);
        if (rc == 0) {
            ++g_launches;
            ++g_tc_launches;
            const long long wn = (long long)I * GH;
            ttg::k_sum_splits<<<(unsigned)((wn / 4 + 255) / 256), 256, 0, st>>>(D.part, ns, wn, wn, D.dwt, accumulate ? 1 : 0);
            ++g_launches;
            if (want_bias) {
                ttg::k_sum_splits<<<(unsigned)((GH / 4 + 255) / 256), 256, 0, st>>>(D.pbias, ns, GH, GH, D.dbias, accumulate ? 1 : 0);
                ++g_launches;
            }
            CU_CHECK(cudaGetLastError());
            return 0;
        }
    }
    const int TMsel = (I <= 64) ? 4 : 8;
    const int BM = 16 * TMsel;
    const int tiles = ((I + BM - 1) / BM) * (GH / ttg::BN);
    // two CTAs per SM are resident: size the split so that the grid fills whole waves (2 waves if possible)
    long long nsplit = (4LL * dv.sms) / tiles;
    if (nsplit < 1) nsplit = 1;
    if (nsplit > kDenseMaxSplit) nsplit = (2LL * dv.sms) / tiles > 0 ? (2LL * dv.sms) / tiles : 1;
    if (nsplit > kDenseMaxSplit) nsplit = kDenseMaxSplit;
    if (nsplit > (rows + 255) / 256) nsplit = (rows + 255) / 256;
    if (nsplit < 1) nsplit = 1;
    ttg::GemmRedArgs g;
    memset(&g, 0, sizeof g);
    g.rows = (unsigned)rows; g.M = I; g.N = GH; g.nsplit = (int)nsplit;
    g.a.p = x; g.a.bstride = x_bstride; g.a.rpb = rpb; g.a.ld = I;
    g.b.p = delta; g.b.bstride = d_bstride; g.b.rpb = rpb; g.b.ld = GH;
    g.part = D.part; g.pbias = want_bias ? D.pbias : nullptr;
    {
        KernelTimer tm(TTRNN_K_GEMM_DW, st);
        if (TMsel == 4) ttg::k_gemm_red<4><<<(unsigned)(tiles * nsplit), ttg::NT, 0, st>>>(g);
        else ttg::k_gemm_red<8><<<(unsigned)(tiles * nsplit), ttg::NT, 0, st>>>(g);
    }
    ++g_launches;
    CU_CHECK(cudaGetLastError());
    const long long wn = (long long)I * GH;
    ttg::k_sum_splits<<<(unsigned)((wn / 4 + 255) / 256), 256, 0, st>>>(D.part, (int)nsplit, wn, wn, D.dwt, accumulate ? 1 : 0);
    ++g_launches;
    if (want_bias) {
        ttg::k_sum_splits<<<(unsigned)((GH / 4 + 255) / 256), 256, 0, st>>>(D.pbias, (int)nsplit, GH, GH, D.dbias, accumulate ? 1 : 0);
        ++g_launches;
    }
    CU_CHECK(cudaGetLastError());
    return 0;
}

// ---- row groups ---------------------------------------------------------------------------------------------------
// A layer-pass of a recurrent kernel is ONE launch of rows / R persistent CTAs that each own R batch rows for all T
// steps, one CTA per SM.  Whenever rows / R is not a multiple of the SM count the launch leaves SMs idle for its whole
// duration (cfg3, 640 rows on 148 SMs: 128 five-row CTAs forward; 148 three-row + 98 two-row CTAs backward), and nothing
// else can use them because layer l + 1 needs layer l of the SAME rows.  Different rows are independent, though: with the
// batch cut into two groups that run the whole stack on two streams, the hardware block scheduler places the CTAs of
// group 1 / layer l beside those of group 0 / layer l + 1, and the SMs stay busy across layer boundaries.  Group 0 is a
// whole number of full waves (sms * m rows), group 1 the remainder.  Each group is a complete, independent call of the
// single-group path on its slice of every row-indexed buffer (own region of `saved` and of the scratch buffers, own
// dense-route GEMMs, own gradient blob, summed at the end), so results do not depend on the split beyond FP32 summation
// order of the parameter gradients.
// per-step gradient logging (log_grads, ttrnn_rnn_backward_logged): (L, B, T, H) buffers the BPTT kernel of layer l writes
// the total gradient of h_t / c_t of every step into; set for the duration of one backward call on this thread
struct StepLog { float *dh = nullptr, *dc = nullptr; long long layer_stride = 0; };
thread_local StepLog t_log;

constexpr int kMaxGroups = 2;
thread_local int t_group = 0;          // group the calling thread is issuing work for (selects the side-stream context)
struct GroupPlan {
    int n = 1;
    long long rows[kMaxGroups] = {0, 0};
};
inline int64_t a256(int64_t bytes) { return (bytes + 255) & ~(int64_t)255; }

struct SimLaunch { int ctas; double dur; };
// Greedy list scheduling of `nq` in-order launch queues on `sms` SMs (one CTA per SM, the earlier-ready launch places its
// CTAs first): the behaviour of the block scheduler with kernels of independent streams.  Returns the makespan.
double sim_makespan(const std::vector<SimLaunch> *q, int nq, int sms) {
    struct Run { double end; int n, s; };
    std::vector<Run> running;
    size_t idx[kMaxGroups] = {};
    int pending[kMaxGroups] = {}, active[kMaxGroups] = {};
    double ready[kMaxGroups] = {};
    for (int s = 0; s < nq; ++s) pending[s] = q[s].empty() ? 0 : q[s][0].ctas;
    int free_sms = sms;
    double t = 0.0;
    for (;;) {
        int order[kMaxGroups];
        for (int s = 0; s < nq; ++s) order[s] = s;
        if (nq == 2 && ready[1] < ready[0]) { order[0] = 1; order[1] = 0; }
        for (int o = 0; o < nq; ++o) {
            const int s = order[o];
            if (idx[s] >= q[s].size() || pending[s] <= 0 || free_sms <= 0) continue;
            const int n = pending[s] < free_sms ? pending[s] : free_sms;
            running.push_back({t + q[s][idx[s]].dur, n, s});
            pending[s] -= n; active[s] += n; free_sms -= n;
        }
        if (running.empty()) break;
        double tmin = running[0].end;
        for (const Run &r : running) if (r.end < tmin) tmin = r.end;
        t = tmin;
        for (size_t i = 0; i < running.size();) {
            if (running[i].end <= t + 1e-9) {
                free_sms += running[i].n; active[running[i].s] -= running[i].n;
                running[i] = running.back(); running.pop_back();
            } else {
                ++i;
            }
        }
        for (int s = 0; s < nq; ++s)
            if (idx[s] < q[s].size() && pending[s] == 0 && active[s] == 0) {
                ++idx[s];
                if (idx[s] < q[s].size()) { pending[s] = q[s][idx[s]].ctas; ready[s] = t; }
            }
    }
    return t;
}

// launches of the recurrent kernels of one group of `Bg` rows: forward layers 0..L-1 into fq, backward L-1..0 into bq.
// Cost of a wave of R rows per CTA ~ (0.4 + R) (measured on the d3r8 chain: forward 2.67 / 4.43 / 6.59 / 10.5 us per step
// at R = 1 / 2 / 3 / 5, backward 2.96 / 4.86 / 7.0 at R = 1 / 2 / 3).  The routes are those of a call on `Bg` rows with
// the kept gates and chunking of the layout `cp.lo`.  false: a layer has no static kernel.
bool group_launches(const CallPlan &cp, long long Bg, std::vector<SimLaunch> *fq, std::vector<SimLaunch> *bq) {
    constexpr double kFloor = 0.4;
    const ttrnn_rnn_desc *d = cp.d();
    const int sms = cp.dv.sms;
    auto push = [&](std::vector<SimLaunch> *q, long long rows, int R) {
        const long long tiles = (rows + R - 1) / R;
        const long long waves = (tiles + sms - 1) / sms;
        q->push_back({(int)(tiles < sms ? tiles : sms), (double)waves * (kFloor + R)});
    };
    for (int l = 0; l < d->num_layers; ++l) {
        const TtsRnnFwdEntry *se = fwd_route(d, cp.rp, l, Bg, sms);
        if (!se) return false;
        push(fq, Bg, se->R);
    }
    for (int l = d->num_layers - 1; l >= 0; --l) {
        BwdRoute br;
        if (bwd_route(d, cp.rp, l, layer_mode(d, l), Bg, sms, cp.lo.kept[l], cp.lo.Tc, &br) || !br.nph) return false;
        for (int q = 0; q < br.nph; ++q) push(bq, br.rows[q], br.e[q]->R);
    }
    return true;
}

// Decide the split.  Only for multi-layer stacks on the static kernels in single-chunk plans (the large-batch configs that
// need time chunks run many waves per launch and lose little to the last one).  Candidates: every cut of the batch at a
// multiple of 4 rows (row-indexed slices stay 16-byte aligned); each side gets the rows-per-CTA variants the single-group
// path would pick for that many rows.  A split is taken when the modelled forward + backward recurrence time drops by
// >= 6 % and the forward alone does not get slower (inference runs the same split).  The search costs a few ms, so the
// result is cached per (descriptor, options, SM count) and host thread.
struct GroupCacheEntry {
    bool used = false;
    ttrnn_rnn_desc d;
    Opts o;
    int sms = 0;
    GroupPlan gp;
};
constexpr int kGroupCache = 16;

int plan_row_groups(const ttrnn_rnn_desc *d_in, GroupPlan *gp, const DevInfo *dev = nullptr) {
    gp->n = 1;
    gp->rows[0] = d_in ? d_in->batch : 0;
    gp->rows[1] = 0;
    if (!d_in || !t_opt.row_groups) return 0;
    if (t_opt.row_groups >= 4) {                        // forced split (tests): group 0 = that many rows, any plan
        const long long r0 = t_opt.row_groups & ~3LL;
        if (r0 < d_in->batch) { gp->n = 2; gp->rows[0] = r0; gp->rows[1] = d_in->batch - r0; }
        return 0;
    }
    if (!t_opt.stat || d_in->num_layers < 2) return 0;
    DevInfo dv;
    if (dev) dv = *dev;
    else if (get_dev(&dv)) return 1;
    thread_local GroupCacheEntry cache[kGroupCache];
    thread_local int cache_next = 0;
    for (const GroupCacheEntry &e : cache)
        if (e.used && e.sms == dv.sms && !memcmp(&e.d, d_in, sizeof *d_in) && !memcmp(&e.o, &t_opt, sizeof t_opt)) {
            *gp = e.gp;
            return 0;
        }
    auto remember = [&]() {
        GroupCacheEntry &e = cache[cache_next];
        cache_next = (cache_next + 1) % kGroupCache;
        e.used = true; e.d = *d_in; e.o = t_opt; e.sms = dv.sms; e.gp = *gp;
        return 0;
    };
    CallPlan cp;
    if (plan_call(d_in, dv, &cp)) return 1;
    const long long B = d_in->batch;
    if (cp.lo.Tc != d_in->seq_len || B < 8 || B > 16LL * dv.sms) return remember();
    std::vector<SimLaunch> f1, b1;
    if (!group_launches(cp, B, &f1, &b1)) return remember();
    const double fwd1 = sim_makespan(&f1, 1, dv.sms), bwd1 = sim_makespan(&b1, 1, dv.sms);
    double best = fwd1 + bwd1;
    const long long step = B <= 1024 ? 4 : 16;
    for (long long r0 = step; r0 < B; r0 += step) {
        std::vector<SimLaunch> fq[kMaxGroups], bq[kMaxGroups];
        if (!group_launches(cp, r0, &fq[0], &bq[0]) || !group_launches(cp, B - r0, &fq[1], &bq[1]))
            continue;
        const double f2 = sim_makespan(fq, 2, dv.sms), b2 = sim_makespan(bq, 2, dv.sms);
        // ties go to the later candidate: the larger group 0 (issued first, on the caller's stream) is the critical path
        if (f2 <= fwd1 * 1.02 && f2 + b2 <= best + 1e-9 && f2 + b2 <= 0.94 * (fwd1 + bwd1)) {
            best = f2 + b2;
            gp->n = 2;
            gp->rows[0] = r0;
            gp->rows[1] = B - r0;
        }
    }
    return remember();
}

// stream + events of the second row group (one per host thread and device, kept for the life of the process)
struct GroupCtx {
    int dev = -1;
    cudaStream_t s = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
};
GroupCtx *group_ctx() {
    thread_local GroupCtx ctx[16];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) return nullptr;
    GroupCtx &c = ctx[dev];
    if (c.dev == dev) return &c;
    if (cudaStreamCreateWithFlags(&c.s, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&c.fork, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&c.join, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    c.dev = dev;
    return &c;
}

}  // namespace

// =============================================================================================
extern "C" {

int ttrnn_abi_version(void) { return TTRNN_ABI_VERSION; }
const char *ttrnn_last_error(void) { return g_err.c_str(); }

int64_t ttrnn_launch_count(int32_t reset) {
    long long v = g_launches.load();
    if (reset) g_launches.store(0);
    return v;
}

int ttrnn_kernel_timing(int32_t enable) {
    g_timing.store(enable ? 1 : 0);
    return 0;
}

int ttrnn_kernel_times(double *ms, int64_t *count) {
    if (!ms || !count) return fail("ms and count must be non-null");
    std::vector<TimedLaunch> recs;
    {
        std::lock_guard<std::mutex> lk(g_time_mu);
        recs.swap(g_timed);
    }
    std::vector<LaunchRecord> out;
    for (auto &r : recs) {
        float t = 0.f;
        if (cudaEventSynchronize(r.b) == cudaSuccess && cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess &&
            r.kind >= 0 && r.kind < TTRNN_K_KINDS) {
            ms[r.kind] += t;
            count[r.kind] += 1;
            out.push_back({r.kind, r.R, r.ctas, r.rows, r.steps, (double)t});
        }
        cudaEventDestroy(r.a);
        cudaEventDestroy(r.b);
    }
    std::lock_guard<std::mutex> lk(g_time_mu);
    g_records.swap(out);
    return 0;
}

int64_t ttrnn_kernel_launch_records(double *buf, int64_t cap_records) {
    std::lock_guard<std::mutex> lk(g_time_mu);
    const int64_t n = (int64_t)g_records.size();
    if (!buf) return n;
    for (int64_t i = 0; i < n && i < cap_records; ++i) {
        const LaunchRecord &r = g_records[i];
        double *o = buf + 6 * i;
        o[0] = r.kind; o[1] = r.R; o[2] = r.ctas; o[3] = (double)r.rows; o[4] = r.steps; o[5] = r.ms;
    }
    return n;
}

int ttrnn_set_option(const char *key, int64_t value) {
    if (!key) return 1;
    if (!strcmp(key, "rows_per_cta")) { g_opt_rows.store(value); return 0; }
    if (!strcmp(key, "chunk_steps")) { g_opt_chunk.store(value); return 0; }
    if (!strcmp(key, "chunk_bytes")) { g_opt_chunk_bytes.store(value > 0 ? value : (4LL << 30)); return 0; }
    if (!strcmp(key, "static_kernels")) { g_opt_static.store(value); return 0; }
    if (!strcmp(key, "save_u_bytes")) { g_opt_save_u_bytes.store(value); return 0; }
    if (!strcmp(key, "static_rows_fwd")) { g_opt_srows_fwd.store(value); return 0; }
    if (!strcmp(key, "static_rows_bwd")) { g_opt_srows_bwd.store(value); return 0; }
    if (!strcmp(key, "row_plan")) { g_opt_row_plan.store(value); return 0; }
    if (!strcmp(key, "gemm_wide")) { g_opt_gemm_wide.store(value); return 0; }
    if (!strcmp(key, "split_kept")) { g_opt_split_kept.store(value); return 0; }
    if (!strcmp(key, "dense_hh_dw")) { g_opt_dense_hh.store(value); return 0; }
    if (!strcmp(key, "dense_ih")) { g_opt_dense_ih.store(value); return 0; }
    if (!strcmp(key, "dense_ih_ratio")) { g_opt_dense_ratio.store(value > 0 ? value : 130); return 0; }
    if (!strcmp(key, "tc_gemm")) { g_opt_tc_gemm.store(value); return 0; }
    if (!strcmp(key, "rank_pad")) { g_opt_rank_pad.store(value); return 0; }
    if (!strcmp(key, "bwd_overlap")) { g_opt_bwd_overlap.store(value); return 0; }
    if (!strcmp(key, "row_groups")) { g_opt_row_groups.store(value); return 0; }
    if (!strcmp(key, "merge_cores")) { g_opt_merge_cores.store(value); return 0; }
    if (!strcmp(key, "tc_red_ts")) { ttc::tc_red_variant() = value ? 1 : 0; return 0; }   // A/B switch, not part of a plan
    if (!strcmp(key, "tc_rows_ts")) { ttc::tc_rows_variant() = value ? 1 : 0; return 0; } // A/B switch, not part of a plan
    return 1;
}

int ttrnn_static_kernel_table(char *buf, int32_t cap) {
    if (!buf || cap < 1) return -1;
    return tts_dump_entries(buf, cap);
}

int ttrnn_rnn_ih_route(const ttrnn_rnn_desc *desc, int32_t layer, int64_t *chain_macs_per_row, int64_t *dense_macs_per_row) {
    t_opt = snapshot_options();
    RnnPlan rp;
    if (build_rnn_plan(desc, &rp)) return -1;
    if (layer < 0 || layer >= desc->num_layers) { fail("layer %d out of range", layer); return -1; }
    const ChainPlan &ih = rp.layer[layer].ih;
    if (chain_macs_per_row) *chain_macs_per_row = chain_macs(ih);
    if (dense_macs_per_row) *dense_macs_per_row = (int64_t)ih.n_in * ih.n_out;
    if (layer == 0 && desc->input_size == 1) return 2;
    return dense_ih_ok(ih, &desc->ih[layer]) ? 1 : 0;
}

int ttrnn_rnn_row_groups(const ttrnn_rnn_desc *desc, int32_t sms, int64_t *rows /*[2]*/) {
    if (!rows) { fail("rows must be non-null"); return -1; }
    t_opt = snapshot_options();
    DevInfo dv;
    if (sms > 0) {
        dv.sms = sms;
        dv.smem_optin = 232448;
        dv.ok = true;
    } else if (get_dev(&dv)) {
        return -1;
    }
    GroupPlan gp;
    if (plan_row_groups(desc, &gp, &dv)) return -1;
    rows[0] = gp.rows[0];
    rows[1] = gp.n == 2 ? gp.rows[1] : 0;
    return gp.n;
}

int64_t ttrnn_tc_launch_count(int32_t reset) {
    long long v = g_tc_launches.load();
    if (reset) g_tc_launches.store(0);
    return v;
}

int ttrnn_rnn_describe(const ttrnn_rnn_desc *d_full, int32_t training, char *buf, int32_t cap) {
    if (!buf || cap < 1) return -1;
    t_opt = snapshot_options();
    // with two row groups the layer lines describe group 0 (the full waves); the header names the split and the
    // rows per CTA the remainder group runs at
    DevInfo dv;
    if (get_dev(&dv)) return -1;
    GroupPlan gp;
    if (plan_row_groups(d_full, &gp, &dv)) return -1;
    ttrnn_rnn_desc d_g0;
    const ttrnn_rnn_desc *d_in = d_full;
    if (gp.n == 2) {
        d_g0 = *d_full;
        d_g0.batch = gp.rows[0];
        d_in = &d_g0;
    }
    CallPlan cp;
    if (plan_call(d_in, dv, &cp)) return -1;
    const ttrnn_rnn_desc *d = cp.d();
    const RnnPlan &rp = cp.rp;
    const RnnLayout &lo = cp.lo;
    const long long B = d->batch;
    const int GH = rp.G * d->hidden_size;
    int n = 0;
    auto put = [&](const char *fmt, ...) {
        if (n >= cap) return;
        va_list ap;
        va_start(ap, fmt);
        n += vsnprintf(buf + n, cap - n, fmt, ap);
        va_end(ap);
    };
    // kernel names as single tokens
    auto tok = [](const char *name) {
        std::string t(name ? name : "none");
        for (auto &c : t)
            if (c == ' ') c = '_';
        return t;
    };
    put("chunk_steps=%d sms=%d tc_gemm=%lld rank_padded=%d bwd_overlap=%d row_groups=%d", lo.Tc, dv.sms, t_opt.tc_gemm,
        (int)cp.eff.padded, lo.overlap, gp.n);
    if (gp.n == 2) {
        std::vector<SimLaunch> fq, bq;
        put(" group_rows0=%lld group_rows1=%lld", gp.rows[0], gp.rows[1]);
        if (group_launches(cp, gp.rows[1], &fq, &bq) && !fq.empty() && !bq.empty())
            put(" group1_fwd_ctas=%d group1_bwd_ctas=%d", fq.back().ctas, bq.front().ctas);
    }
    put("\n");
    for (int l = 0; l < d->num_layers; ++l) {
        const LayerPlan &lp = rp.layer[l];
        const int mode = layer_mode(d, l);
        const bool rank1 = mode == tts::MODE_RANK1;
        const bool dense = !rank1 && dense_ih_ok(lp.ih, &d->ih[l]);
        const char *route = rank1 ? "rank_one" : (dense ? "dense" : "tt_chain");
        const bool tc_f = dense && tc_rows_use(B * (long long)lo.Tc, lp.ih.n_in, GH, false);
        const bool tc_r = dense && t_opt.tc_gemm && ttc::tc_red_ok(B * (long long)lo.Tc, lp.ih.n_in, GH);
        const TtsRnnFwdEntry *se = fwd_route(d, rp, l, B, dv.sms);
        // save_mode 2 = kept gate activations, 0 = recompute
        put("layer=%d ih_route=%s ih_fwd_tc=%d ih_dw_tc=%d fwd_kernel=%s fwd_rows=%d save_mode=%d", l, route, (int)tc_f, (int)tc_r,
            se ? tok(se->name).c_str() : "runtime", se ? se->R : 0, lo.kept[l] ? 2 : 0);
        if (training) {
            BwdRoute br;
            if (bwd_route(d, rp, l, mode, B, dv.sms, lo.kept[l], lo.Tc, &br)) return -1;
            if (!br.nph) {
                put(" bwd_kernel=runtime bwd_rows=0");
            } else {
                put(" bwd_kernel=%s bwd_rows=%d bwd_phase_rows=%lld", tok(br.e[0]->name).c_str(), br.e[0]->R, br.rows[0]);
                if (br.nph == 2)
                    put(" bwd_kernel2=%s bwd_rows2=%d bwd_phase_rows2=%lld", tok(br.e[1]->name).c_str(), br.e[1]->R, br.rows[1]);
                put(" hh_dw=%s hh_dw_tc=%d", br.split ? (br.dense_hh ? "dense" : "tt_chain") : "fused",
                    (int)(br.dense_hh && t_opt.tc_gemm && ttc::tc_red_ok(B * (long long)lo.Tc, d->hidden_size, GH)));
            }
        }
        put("\n");
    }
    return n;
}

int64_t ttrnn_rnn_param_count(const ttrnn_rnn_desc *desc) {
    RnnPlan rp;
    if (build_rnn_plan(desc, &rp)) return -1;
    return rp.param_floats;
}

int64_t ttrnn_rnn_param_count_proj(const ttrnn_rnn_desc *desc, const ttrnn_rnn_proj *pj) {
    if (!pj) { fail("ttrnn_rnn_param_count_proj: pj must be non-null"); return -1; }
    RnnPlan rp;
    if (build_rnn_plan(desc, &rp, pj)) return -1;
    return rp.param_floats;
}

// byte sizes of ONE row group (the whole batch when the plan has a single group), under the calling thread's options
static int workspace_one(const ttrnn_rnn_desc *desc, ttrnn_rnn_workspace *ws, bool keep_masked,
                         const ttrnn_rnn_proj *pj = nullptr) {
    DevInfo dv;
    CallPlan cp;
    if (get_dev(&dv) || plan_call(desc, dv, &cp, keep_masked, pj)) return 1;
    ws->saved_bytes = cp.lo.sv_total * 4;
    ws->fwd_scratch_bytes = (cp.lo.f_total + cp.eff.pad_floats) * 4;       // + the rank-padded parameter blob
    ws->bwd_scratch_bytes = (cp.lo.b_total + 2 * cp.eff.pad_floats) * 4;   // + padded parameters and padded gradients
    return 0;
}

int ttrnn_rnn_workspace_bytes(const ttrnn_rnn_desc *desc, ttrnn_rnn_workspace *ws) {
    return ttrnn_rnn_workspace_bytes_ex(desc, 0, ws);
}

int ttrnn_rnn_workspace_bytes_ex(const ttrnn_rnn_desc *desc, int32_t flags, ttrnn_rnn_workspace *ws) {
    if (!ws) return fail("null workspace struct");
    if (flags & TTRNN_WS_PROJ) return fail("TTRNN_WS_PROJ: size the plan with ttrnn_rnn_workspace_bytes_proj");
    t_opt = snapshot_options();
    if (flags & TTRNN_WS_WHOLE_BATCH) t_opt.row_groups = 0;
    GroupPlan gp;
    if (plan_row_groups(desc, &gp)) return 1;
    const bool masked = (flags & TTRNN_WS_DROPOUT) != 0;
    if (gp.n == 1) {
        if (workspace_one(desc, ws, masked)) return 1;
    } else {
        // one region per group in every buffer (256-byte aligned), + the gradient blob of every group but the first
        const int64_t pf = ttrnn_rnn_param_count(desc);
        ws->saved_bytes = ws->fwd_scratch_bytes = ws->bwd_scratch_bytes = 0;
        for (int g = 0; g < gp.n; ++g) {
            ttrnn_rnn_desc dg = *desc;
            dg.batch = gp.rows[g];
            ttrnn_rnn_workspace wg;
            if (workspace_one(&dg, &wg, masked)) return 1;
            ws->saved_bytes += a256(wg.saved_bytes);
            ws->fwd_scratch_bytes += a256(wg.fwd_scratch_bytes);
            ws->bwd_scratch_bytes += a256(wg.bwd_scratch_bytes) + (g > 0 ? a256(pf * 4) : 0);
        }
    }
    memset(ws->plan, 0, sizeof ws->plan);
    plan_store(t_opt, ws->plan);
    ws->plan[kPlanGroups] = gp.n;
    ws->plan[kPlanRows0] = gp.rows[0];
    ws->plan[kPlanLayerStates] = (flags & TTRNN_WS_LAYER_STATES) ? 1 : 0;
    ws->plan[kPlanDropout] = masked ? 1 : 0;
    return 0;
}

// a projected stack runs as one row group: the group split is planned from the static kernels, which it has none of
int ttrnn_rnn_workspace_bytes_proj(const ttrnn_rnn_desc *desc, const ttrnn_rnn_proj *pj, int32_t flags,
                                   ttrnn_rnn_workspace *ws) {
    if (!ws) return fail("null workspace struct");
    if (!pj) return fail("ttrnn_rnn_workspace_bytes_proj: pj must be non-null");
    if (!desc) return fail("null descriptor");
    if (desc->cell != TTRNN_CELL_LSTM) return fail("ttrnn_rnn_workspace_bytes_proj: a projection needs an LSTM descriptor");
    t_opt = snapshot_options();
    t_opt.row_groups = 0;
    const bool masked = (flags & TTRNN_WS_DROPOUT) != 0;
    if (workspace_one(desc, ws, masked, pj)) return 1;
    memset(ws->plan, 0, sizeof ws->plan);
    plan_store(t_opt, ws->plan);
    ws->plan[kPlanGroups] = 1;
    ws->plan[kPlanRows0] = desc->batch;
    ws->plan[kPlanLayerStates] = (flags & TTRNN_WS_LAYER_STATES) ? 1 : 0;
    ws->plan[kPlanDropout] = masked ? 1 : 0;
    ws->plan[kPlanProj] = 1;
    return 0;
}

// forward of ONE row group on stream `stream`; `ws` carries the byte sizes of this group, t_opt is already loaded
// `dc`: inter-layer dropout (nullptr = none; the plan then has no masked buffers)
// `pj`: the projection (nullptr = none)
static int forward_one(const ttrnn_rnn_desc *d_in, const ttrnn_rnn_workspace *ws, const StateMap &sm, const float *x,
                       const float *h0, const float *c0, const float *params_in, float *out, float *hT, float *cT, void *saved,
                       void *scratch, void *stream, const DropCall *dc, const ttrnn_rnn_proj *pj) {
    if (!x || !params_in || !out || !scratch) return fail("x, params, out and scratch must be non-null");
    DevInfo dv;
    CallPlan cp;
    if (get_dev(&dv) || plan_call(d_in, dv, &cp, ws->plan[kPlanDropout] != 0, pj)) return 1;
    const ttrnn_rnn_desc *d = cp.d();
    const RnnPlan &rp = cp.rp;
    const RnnLayout &lo = cp.lo;
    const EffDesc &eff = cp.eff;
    if ((lo.f_total + eff.pad_floats) * 4 != ws->fwd_scratch_bytes || lo.sv_total * 4 != ws->saved_bytes)
        return fail("ttrnn_rnn_forward: workspace struct does not belong to this descriptor (scratch %lld vs %lld bytes)",
                    (long long)(lo.f_total + eff.pad_floats) * 4, (long long)ws->fwd_scratch_bytes);
    cudaStream_t st = (cudaStream_t)stream;
    const float *params = params_in;
    if (eff.padded) {
        // rank-padded copy of the parameter blob (zeros on the added rank slices)
        float *pp = (float *)scratch + lo.f_total;
        CU_CHECK(cudaMemsetAsync(pp, 0, (size_t)eff.pad_floats * 4, st));
        k_pad_cores<<<eff.tab.n, 256, 0, st>>>(eff.tab, params_in, pp);
        ++g_launches;
        CU_CHECK(cudaGetLastError());
        params = pp;
    }
    const long long B = d->batch;
    const int T = d->seq_len, H = d->hidden_size, L = d->num_layers, G = rp.G;
    const int GH = G * H, W = rp.out_width(d);       // W: width of a layer's output and h state
    const bool lstm = d->cell == TTRNN_CELL_LSTM;
    float *sc = (float *)scratch;
    float *sv = (float *)saved;
    float *xg = sc + lo.f_xg;
    float *st_h = sc + lo.f_sh, *st_c = sc + lo.f_sc;

    for (int l = 0; l < L; ++l) {
        const LayerPlan &lp = rp.layer[l];
        const int nin = lp.ih.n_in;
        const float *lin;       // input of this layer (B, T, nin)
        if (l == 0) lin = x;
        else lin = sv ? sv + lo.sv_hs + (long long)(l - 1) * lo.BTW : sc + lo.f_hs + ((l - 1) & 1) * r4(lo.BTW);
        if (l > 0 && dc) {
            // dropout: layer l reads the masked output of layer l - 1 (kept for the backward in training)
            float *masked = sv ? sv + lo.sv_drop + (long long)(l - 1) * lo.BTW : sc + lo.f_drop;
            if (launch_dropout(dv, B, T, W, *dc, dc->row0, l - 1, lin, nullptr, masked, nullptr, st)) return 1;
            lin = masked;
        }
        float *lout;            // output of this layer (B, T, W)
        if (l == L - 1) lout = out;
        else lout = sv ? sv + lo.sv_hs + (long long)l * lo.BTW : sc + lo.f_hs + (l & 1) * r4(lo.BTW);
        float *csave = (sv && lstm) ? sv + lo.sv_cs + (long long)l * lo.BTH : nullptr;
        const float *b_ih = d->has_bias ? params + lp.off_ih_bias : nullptr;
        const float *b_hh = d->has_bias ? params + lp.off_hh_bias : nullptr;
        // this layer's initial state, read by its first chunk, and where its last chunk leaves the final state
        const float *h0l = sm.init(h0, l), *c0l = sm.init(c0, l, true);
        float *hTl = sm.fin(hT, l, L), *cTl = sm.fin(cT, l, L, true);

        // ---- batched ih projection of one time chunk: xg[b, t, :] = W_ih x[b, t0+t, :] + b_ih (+ b_hh for LSTM),
        // through the TT chain or, when that is the cheaper contraction order, through dense W_ih^T
        const int mode = layer_mode(d, l);
        const bool dense = mode == tts::MODE_XG && dense_ih_ok(lp.ih, &d->ih[l]);
        DenseIh D;
        if (dense) {
            dense_carve(sc + lo.f_dense, lp.ih, false, &D);
            if (dense_prepare(lp.ih, &d->ih[l], dv, params + lp.off_ih_cores, D, false,
                              tc_rows_use(B * (long long)lo.Tc, nin, GH, false), false, st))
                return 1;
        }
        auto project = [&](int t0, int tc) -> int {
            if (dense)
                return dense_rows_gemm(TTRNN_K_GEMM_FWD, dv, B * tc, tc, lin + (long long)t0 * nin, (long long)T * nin, nin,
                                       D.wt, D.w_hi, D.w_lo, GH, b_ih, lstm ? b_hh : nullptr, xg, (long long)tc * GH, false, st);
            return launch_ttlinear_fwd(lp.ih, dv, B * tc, tc, lin + (long long)t0 * nin, (long long)T * nin,
                                       params + lp.off_ih_cores, b_ih, lstm ? b_hh : nullptr, xg, (long long)tc * GH, st,
                                       &d->ih[l]);
        };

        // ---- statically specialised kernel for this hh shape, if one is registered -------------------
        const TtsRnnFwdEntry *se = fwd_route(d, rp, l, B, dv.sms);
        if (se) {
            int occ = 0;
            int rc = se->prepare(&occ);
            if (rc || occ < 1) return fail("static kernel %s cannot be configured (cuda error %d)", se->name, rc);
            long long g = (long long)occ * dv.sms;
            const long long tiles = (B + se->R - 1) / se->R;
            if (g > tiles) g = tiles;
            tts::RnnFwdSArgs sa;
            memset(&sa, 0, sizeof sa);
            sa.B = B;
            sa.cores = params + lp.off_hh_cores;
            float *aux = sc + lo.f_aux;
            if (mode == tts::MODE_RANK1) {
                // W_ih has a single column: densify it once (the TT chain applied to the scalar 1)
                k_fill<<<1, 32, 0, st>>>(aux + r4(GH), 1.0f, 1);
                ++g_launches;
                if (launch_ttlinear_fwd(lp.ih, dv, 1, 1, aux + r4(GH), 0, params + lp.off_ih_cores, nullptr, nullptr,
                                        aux, 0, st))
                    return 1;
                sa.w_eff = aux;
                sa.bias_ih = b_ih;
                sa.bias_hh = b_hh;
            } else {
                sa.bias_hh = lstm ? nullptr : b_hh;
            }
            const int chunk = (mode == tts::MODE_RANK1) ? T : lo.Tc;
            for (int t0 = 0; t0 < T; t0 += chunk) {
                const int tc = (T - t0 < chunk) ? T - t0 : chunk;
                if (mode == tts::MODE_XG) {
                    if (project(t0, tc)) return 1;
                    sa.xg = xg; sa.xg_bstride = (long long)tc * GH;
                } else {
                    sa.x1 = lin + t0; sa.x1_bstride = T;
                }
                const bool first = (t0 == 0), last = (t0 + tc == T);
                sa.steps = tc;
                sa.h_in = first ? h0l : st_h;
                sa.c_in = first ? c0l : st_c;
                sa.out = lout + (long long)t0 * H; sa.out_bstride = (long long)T * H;
                sa.c_save = csave ? csave + (long long)t0 * H : nullptr;
                if (sv && lo.kept[l]) {
                    sa.u_save = sv + lo.sv_u[l] + (long long)t0 * 4 * H;       sa.u_bstride = (long long)T * 4 * H;
                }
                sa.h_out = (last && hTl) ? hTl : st_h;
                sa.c_out = (last && cTl) ? cTl : st_c;
                {
                    KernelTimer tm(TTRNN_K_RNN_FWD, st, se->R, (int)g, B, tc);
                    rc = se->launch(&sa, (int)g, st);
                }
                ++g_launches;
                if (rc) return fail("static kernel %s launch failed: %s", se->name, cudaGetErrorString((cudaError_t)rc));
            }
            continue;
        }

        if (rp.P) {
            // projected LSTM: the projection chain runs inside the recurrent kernel after the gate math of every step
            RnnFwdProjArgs a;
            memset(&a, 0, sizeof a);
            a.p = lp.hh;
            a.q = lp.hr;
            const int R = pick_rows([&](int r) { return smem_rnn_fwd_proj(lp.hh, lp.hr, r, H); }, dv.smem_optin, 8, B,
                                    dv.sms, 2);
            if (R == 0)
                return fail("layer %d: projected hh / hr TT shapes need %lld bytes of shared memory per CTA (limit %d): "
                            "unsupported", l, smem_rnn_fwd_proj(lp.hh, lp.hr, 1, H) * 4, dv.smem_optin);
            a.R = R;
            fill_tiles(lp.hh, R, a.tile, nullptr, nullptr);
            fill_tiles(lp.hr, R, a.tile_q, nullptr, nullptr);
            a.H = H; a.P = W; a.B = B;
            a.cores = params + lp.off_hh_cores;
            a.cores_q = params + lp.off_hr_cores;
            const size_t smem = (size_t)smem_rnn_fwd_proj(lp.hh, lp.hr, R, H) * 4;
            int grid = 0;
            if (grid_for(k_rnn_fwd_proj, smem, (B + R - 1) / R, dv, &grid)) return 1;
            for (int t0 = 0; t0 < T; t0 += lo.Tc) {
                const int tc = (T - t0 < lo.Tc) ? T - t0 : lo.Tc;
                if (project(t0, tc)) return 1;
                const bool first = (t0 == 0), last = (t0 + tc == T);
                a.steps = tc;
                a.xg = xg; a.xg_bstride = (long long)tc * GH;
                a.h_in = first ? h0l : st_h;
                a.c_in = first ? c0l : st_c;
                a.out = lout + (long long)t0 * W; a.out_bstride = (long long)T * W;
                a.c_save = csave ? csave + (long long)t0 * H : nullptr; a.c_bstride = (long long)T * H;
                a.h_out = (last && hTl) ? hTl : st_h;
                a.c_out = (last && cTl) ? cTl : st_c;
                {
                    KernelTimer tm(TTRNN_K_RNN_FWD, st, R, grid, B, tc);
                    k_rnn_fwd_proj<<<grid, TT_NTHREADS, smem, st>>>(a);
                }
                ++g_launches;
                CU_CHECK(cudaGetLastError());
            }
            continue;
        }

        // recurrent kernel configuration for this layer
        RnnFwdArgs a;
        memset(&a, 0, sizeof a);
        a.p = lp.hh;
        const int R = pick_rows([&](int r) { return smem_rnn_fwd(lp.hh, r, H, G); }, dv.smem_optin, 8, B, dv.sms, 2);
        if (R == 0)
            return fail("layer %d: hh TT shape needs %lld bytes of shared memory per CTA (limit %d): unsupported", l,
                        smem_rnn_fwd(lp.hh, 1, H, G) * 4, dv.smem_optin);
        a.R = R;
        fill_tiles(lp.hh, R, a.tile, nullptr, nullptr);
        a.cell = d->cell; a.H = H; a.G = G; a.B = B;
        a.cores = params + lp.off_hh_cores;
        a.bias_hh = lstm ? nullptr : b_hh;
        const size_t smem = (size_t)smem_rnn_fwd(lp.hh, R, H, G) * 4;
        int grid = 0;
        if (grid_for(k_rnn_fwd, smem, (B + R - 1) / R, dv, &grid)) return 1;

        for (int t0 = 0; t0 < T; t0 += lo.Tc) {
            const int tc = (T - t0 < lo.Tc) ? T - t0 : lo.Tc;
            // (1) batched ih projection of the chunk
            if (project(t0, tc)) return 1;
            // (2) persistent recurrence over the chunk
            const bool first = (t0 == 0), last = (t0 + tc == T);
            a.steps = tc;
            a.xg = xg; a.xg_bstride = (long long)tc * GH;
            a.h_in = first ? h0l : st_h;
            a.c_in = first ? c0l : st_c;
            a.out = lout + (long long)t0 * H; a.out_bstride = (long long)T * H;
            a.c_save = csave ? csave + (long long)t0 * H : nullptr;
            a.h_out = (last && hTl) ? hTl : st_h;
            a.c_out = (last && cTl) ? cTl : st_c;
            {
                KernelTimer tm(TTRNN_K_RNN_FWD, st, R, grid, B, tc);
                k_rnn_fwd<<<grid, TT_NTHREADS, smem, st>>>(a);
            }
            ++g_launches;
            CU_CHECK(cudaGetLastError());
        }
    }
    return 0;
}

// second stream + events of the backward overlap (one per host thread and device; created on first use, kept for the
// life of the process).  Events carry no timing so that recording them is cheap.
struct SideCtx {
    int dev = -1;
    cudaStream_t s = nullptr;
    cudaEvent_t fork = nullptr, fin = nullptr, done[2] = {nullptr, nullptr};
};
static SideCtx *side_ctx() {
    thread_local SideCtx ctx[16][kMaxGroups];      // every row group forks its own side stream
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) return nullptr;
    SideCtx &c = ctx[dev][t_group];
    if (c.dev == dev) return &c;
    if (cudaStreamCreateWithFlags(&c.s, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&c.fork, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&c.fin, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    for (int i = 0; i < 2; ++i)
        if (cudaEventCreateWithFlags(&c.done[i], cudaEventDisableTiming) != cudaSuccess) return nullptr;
    c.dev = dev;
    return &c;
}

// body of ttrnn_rnn_backward on the effective (possibly rank-padded) descriptor
static int rnn_backward_impl(const CallPlan &cp, const StateMap &sm, const float *x, const float *h0, const float *c0,
                             const float *params, const float *out, const void *saved, const float *d_out, const float *d_hT,
                             const float *d_cT, float *d_params, float *d_x, float *d_h0, float *d_c0, void *scratch,
                             cudaStream_t st, const DropCall *dc);

static int backward_one(const ttrnn_rnn_desc *d_in, const ttrnn_rnn_workspace *ws, const StateMap &sm, const float *x,
                        const float *h0, const float *c0, const float *params, const float *out, const void *saved,
                        const float *d_out, const float *d_hT, const float *d_cT, float *d_params, float *d_x, float *d_h0,
                        float *d_c0, void *scratch, void *stream, const DropCall *dc, const ttrnn_rnn_proj *pj) {
    if (!x || !params || !out || !scratch || !d_params) return fail("x, params, out, scratch, d_params must be non-null");
    DevInfo dv;
    CallPlan cp;
    if (get_dev(&dv) || plan_call(d_in, dv, &cp, ws->plan[kPlanDropout] != 0, pj)) return 1;
    const RnnLayout &lo = cp.lo;
    const EffDesc &eff = cp.eff;
    if ((lo.b_total + 2 * eff.pad_floats) * 4 != ws->bwd_scratch_bytes || lo.sv_total * 4 != ws->saved_bytes)
        return fail("ttrnn_rnn_backward: workspace struct does not belong to this descriptor (scratch %lld vs %lld bytes)",
                    (long long)(lo.b_total + 2 * eff.pad_floats) * 4, (long long)ws->bwd_scratch_bytes);
    cudaStream_t st = (cudaStream_t)stream;
    if (!eff.padded)
        return rnn_backward_impl(cp, sm, x, h0, c0, params, out, saved, d_out, d_hT, d_cT, d_params, d_x, d_h0, d_c0, scratch,
                                 st, dc);
    float *pp = (float *)scratch + lo.b_total, *dpp = pp + eff.pad_floats;
    CU_CHECK(cudaMemsetAsync(pp, 0, (size_t)eff.pad_floats * 4, st));
    k_pad_cores<<<eff.tab.n, 256, 0, st>>>(eff.tab, params, pp);
    ++g_launches;
    CU_CHECK(cudaGetLastError());
    if (rnn_backward_impl(cp, sm, x, h0, c0, pp, out, saved, d_out, d_hT, d_cT, dpp, d_x, d_h0, d_c0, scratch, st, dc)) return 1;
    // the gradient wrt a real core is the matching block of the padded core's gradient
    k_unpad_cores<<<eff.tab.n, 256, 0, st>>>(eff.tab, dpp, d_params);
    ++g_launches;
    CU_CHECK(cudaGetLastError());
    return 0;
}

static int rnn_backward_impl(const CallPlan &cp, const StateMap &sm, const float *x, const float *h0, const float *c0,
                             const float *params, const float *out, const void *saved, const float *d_out, const float *d_hT,
                             const float *d_cT, float *d_params, float *d_x, float *d_h0, float *d_c0, void *scratch,
                             cudaStream_t st, const DropCall *dc) {
    const ttrnn_rnn_desc *d = cp.d();
    const RnnPlan &rp = cp.rp;
    const RnnLayout &lo = cp.lo;
    const DevInfo &dv = cp.dv;
    const long long B = d->batch;
    const int T = d->seq_len, H = d->hidden_size, L = d->num_layers, G = rp.G;
    const int GH = G * H, W = rp.out_width(d);       // W: width of a layer's output and h state
    const bool lstm = d->cell == TTRNN_CELL_LSTM;
    if ((L > 1 || lstm) && !saved) return fail("backward needs the `saved` buffer written by a training forward");
    if (dc && L > 1 && !lo.masked) return fail("internal: dropout backward without the masked layer inputs");
    float *sc = (float *)scratch;
    const float *sv = (const float *)saved;
    float *sdh = sc + lo.b_sdh, *sdc = sc + lo.b_sdc;
    // backward overlap (build_layout): two sets of the per-layer buffers; `side` runs the deferred weight-gradient work
    SideCtx *side = lo.overlap ? side_ctx() : nullptr;
    bool set_busy[2] = {false, false};
    // every exit path must give the caller's stream the side work back
    struct Join {
        SideCtx *side; cudaStream_t st; bool used;
        ~Join() {
            if (!side || !used) return;
            cudaEventRecord(side->fin, side->s);
            cudaStreamWaitEvent(st, side->fin, 0);
        }
    } join{side, st, false};

    for (int l = L - 1; l >= 0; --l) {
        const LayerPlan &lp = rp.layer[l];
        const int nin = lp.ih.n_in;
        const int set = lo.overlap ? (l & 1) : 0;
        float *ss = sc + (long long)set * lo.set_stride;      // this layer's buffer set
        if (side && set_busy[set]) {                          // layer l + 2 used the same set
            CU_CHECK(cudaStreamWaitEvent(st, side->done[set], 0));
            set_busy[set] = false;
        }
        float *xg = ss + lo.b_xg;
        float *part_hh = ss + lo.b_part_hh, *part_ih = ss + lo.b_part_ih;
        cudaStream_t ws = st;                                 // stream of the weight-gradient work of this layer
        DevInfo dvw = dv;                                     // ... and the SMs it may plan for
        // dropout: layers >= 1 read the masked output of the layer below, which the forward kept
        const float *lin = (l == 0) ? x : sv + (dc ? lo.sv_drop : lo.sv_hs) + (long long)(l - 1) * lo.BTW;
        const float *lout = (l == L - 1) ? out : sv + lo.sv_hs + (long long)l * lo.BTW;
        const float *lcs = lstm ? sv + lo.sv_cs + (long long)l * lo.BTH : nullptr;
        // gradient wrt this layer's outputs / wrt its inputs
        const float *dhs = (l == L - 1) ? d_out : sc + lo.b_dhs + ((l + 1) & 1) * r4(lo.BTW);
        float *dlin = (l == 0) ? d_x : sc + lo.b_dhs + (l & 1) * r4(lo.BTW);
        if (l < L - 1 && dc) {
            // dropout: the gradient wrt the masked input of layer l + 1 (its dX, written on this stream also under the
            // backward overlap) times mask / (1 - p) is the gradient wrt this layer's output; in place
            float *g = sc + lo.b_dhs + ((l + 1) & 1) * r4(lo.BTW);
            if (launch_dropout(dv, B, T, W, *dc, dc->row0, l, g, nullptr, g, nullptr, st)) return 1;
        }
        const float *b_ih = d->has_bias ? params + lp.off_ih_bias : nullptr;
        const float *b_hh = d->has_bias ? params + lp.off_hh_bias : nullptr;
        // this layer's initial state and the upstream gradient of its final state (enters its last step)
        const float *h0l = sm.init(h0, l), *c0l = sm.init(c0, l, true);
        const float *dhTl = sm.fin(d_hT, l, L), *dcTl = sm.fin(d_cT, l, L, true);

        // ---- ih projection (recompute) and its backward per time chunk: TT chain or dense route ---------
        // a rank-one layer 0 whose input gradient is wanted runs the projected-input kernels (delta_ih feeds dX)
        const int mode = d_x ? tts::MODE_XG : layer_mode(d, l);
        const bool dense = mode == tts::MODE_XG && dense_ih_bwd_ok(lp.ih, dlin != nullptr, &d->ih[l]);
        DenseIh D;
        if (dense) {
            dense_carve(ss + lo.b_dense, lp.ih, true, &D);
            if (dense_prepare(lp.ih, &d->ih[l], dv, params + lp.off_ih_cores, D, dlin != nullptr,
                              tc_rows_use(B * (long long)lo.Tc, nin, GH, false),
                              dlin != nullptr && tc_rows_use(B * (long long)lo.Tc, GH, nin, true), st))
                return 1;
        }
        bool dense_first = true;
        auto project = [&](int t0, int tc) -> int {
            if (dense)
                return dense_rows_gemm(TTRNN_K_GEMM_FWD, dv, B * tc, tc, lin + (long long)t0 * nin, (long long)T * nin, nin,
                                       D.wt, D.w_hi, D.w_lo, GH, b_ih, lstm ? b_hh : nullptr, xg, (long long)tc * GH, false, st);
            return launch_ttlinear_fwd(lp.ih, dv, B * tc, tc, lin + (long long)t0 * nin, (long long)T * nin,
                                       params + lp.off_ih_cores, b_ih, lstm ? b_hh : nullptr, xg, (long long)tc * GH, st,
                                       &d->ih[l]);
        };
        // xg holds delta_ih of the chunk: core / bias gradients (accumulated over chunks) and dX
        auto project_dx = [&](int t0, int tc) -> int {       // dense route: dX = delta W on the caller's stream
            return dense_rows_gemm(TTRNN_K_GEMM_DX, dv, B * tc, tc, xg, (long long)tc * GH, GH, D.w, D.wt_hi, D.wt_lo, nin,
                                   nullptr, nullptr, dlin + (long long)t0 * nin, (long long)T * nin, true, st);
        };
        bool dx_done = false;                                 // overlap: dX was issued before the fork
        auto project_bwd = [&](int t0, int tc, int *ih_used) -> int {
            if (dense) {
                if (dense_dw(dvw, B * tc, tc, lin + (long long)t0 * nin, (long long)T * nin, nin, xg, (long long)tc * GH, GH,
                             D, !dense_first, d->has_bias != 0, ws))
                    return 1;
                dense_first = false;
                if (dlin && !dx_done) return project_dx(t0, tc);
                return 0;
            }
            return launch_ttlinear_bwd(lp.ih, dv, B * tc, tc, lin + (long long)t0 * nin, (long long)T * nin,
                                       params + lp.off_ih_cores, xg, (long long)tc * GH,
                                       dlin ? dlin + (long long)t0 * nin : nullptr, (long long)T * nin, part_ih,
                                       lo.nslots, ss + lo.b_spill, 1, st, ih_used, &d->ih[l]);
        };
        // after the last chunk: dense dW^T -> TT cores (I-row TT-matvec backward on the identity), bias copy
        auto project_finish = [&](int *ih_used) -> int {
            if (!dense) return 0;
            if (launch_ttlinear_bwd(lp.ih, dvw, nin, nin, D.eye, 0, params + lp.off_ih_cores, D.dwt, 0, nullptr, 0, part_ih,
                                    lo.nslots, ss + lo.b_spill, 0, ws, ih_used, &d->ih[l]))
                return 1;
            return 0;
        };

        // ---- statically specialised BPTT kernel for this hh shape, if one is registered ---------------
        // per-step gradient logging is emitted by the runtime-shape BPTT kernel (it recomputes from hs / cs, which every
        // training forward keeps, so it can follow a forward that ran on the static kernels).  Where the forward kept the
        // gate activations of this layer, the route prefers the kernels that consume them.
        const bool logging = t_log.dh != nullptr;
        BwdRoute br;
        if (!logging && bwd_route(d, rp, l, mode, B, dv.sms, lo.kept[l] && sv, lo.Tc, &br)) return 1;
        if (br.nph) {
            const bool split = br.split, split_r1 = br.split_r1, dense_hh = br.dense_hh;
            int ph_grid[2] = {0, 0};
            int rc = 0;
            int sgrid = 0;
            for (int q = 0; q < br.nph; ++q) {
                int occ = 0;
                rc = br.e[q]->prepare(&occ);
                if (rc || occ < 1) return fail("static kernel %s cannot be configured (cuda error %d)", br.e[q]->name, rc);
                long long g = (long long)occ * dv.sms;
                const long long tiles = (br.rows[q] + br.e[q]->R - 1) / br.e[q]->R;
                if (g > tiles) g = tiles;
                if (g > lo.nslots) g = lo.nslots;
                ph_grid[q] = (int)g;
                if (ph_grid[q] > sgrid) sgrid = ph_grid[q];
            }
            // launch every phase of the plan on its rows (row-indexed pointers are offset; gradient slots are shared
            // and accumulated: the phases run back to back on the stream)
            auto launch_plan = [&](const tts::RnnBwdSArgs &base) -> int {
                for (int q = 0; q < br.nph; ++q) {
                    tts::RnnBwdSArgs a2 = base;
                    const long long r0 = br.row0[q];
                    a2.B = br.rows[q];
                    if (a2.xg) a2.xg += r0 * a2.xg_bstride;
                    if (a2.x1) a2.x1 += r0 * a2.x1_bstride;
                    if (a2.hs) a2.hs += r0 * (long long)T * H;
                    if (a2.cs) a2.cs += r0 * (long long)T * H;
                    if (a2.dhs) a2.dhs += r0 * (long long)T * H;
                    if (a2.h0) a2.h0 += r0 * H;
                    if (a2.c0) a2.c0 += r0 * H;
                    if (a2.dh_in) a2.dh_in += r0 * H;
                    if (a2.dc_in) a2.dc_in += r0 * H;
                    if (a2.dh_out) a2.dh_out += r0 * H;
                    if (a2.dc_out) a2.dc_out += r0 * H;
                    if (a2.u_save) a2.u_save += r0 * a2.u_bstride;
                    int e;
                    {
                        KernelTimer tm(TTRNN_K_RNN_BWD, st, br.e[q]->R, ph_grid[q], br.rows[q], a2.steps);
                        e = br.e[q]->launch(&a2, ph_grid[q], st);
                    }
                    ++g_launches;
                    if (e) return fail("static kernel %s launch failed: %s", br.e[q]->name, cudaGetErrorString((cudaError_t)e));
                }
                return 0;
            };
            const long long slot = br.e[0]->slot_floats;
            if (slot > lo.part_stride) return fail("internal: gradient slot too small");
            const long long ih_slot = lp.ih.core_floats + GH;
            const long long hhw_slot = lp.hh.core_floats + GH;       // slot layout of the batched hh-dW kernel (split mode)
            int hh_used = 0;
            CU_CHECK(cudaMemsetAsync(part_hh, 0, (size_t)((split && !split_r1) ? hhw_slot * lo.nslots : slot * sgrid) * 4, st));
            CU_CHECK(cudaMemsetAsync(part_ih, 0, (size_t)ih_slot * lo.nslots * 4, st));
            tts::RnnBwdSArgs sa;
            memset(&sa, 0, sizeof sa);
            sa.B = B; sa.T = T;
            sa.cores = params + lp.off_hh_cores;
            sa.hs = lout; sa.cs = lcs; sa.h0 = h0l; sa.c0 = c0l; sa.dhs = dhs;
            sa.partial = (split && !split_r1) ? nullptr : part_hh;
            if (br.kept) { sa.u_save = sv + lo.sv_u[l]; sa.u_bstride = (long long)T * 4 * H; }
            float *aux = ss + lo.b_aux;
            float *aux_g = aux + r4(GH);
            float *one = aux_g + r4(GH);
            int ih_used = 0;
            DenseIh DH;
            int hh_dense_calls = 0;
            if (dense_hh) {
                dense_carve(ss + lo.b_dense_hh, lp.hh, true, &DH);
                ttg::k_eye<<<1024, 256, 0, st>>>(DH.eye, H);
                ++g_launches;
                CU_CHECK(cudaGetLastError());
            }
            if (mode == tts::MODE_RANK1) {
                k_fill<<<1, 32, 0, st>>>(one, 1.0f, 1);
                ++g_launches;
                if (launch_ttlinear_fwd(lp.ih, dv, 1, 1, one, 0, params + lp.off_ih_cores, nullptr, nullptr, aux, 0, st))
                    return 1;
                sa.w_eff = aux; sa.bias_ih = b_ih; sa.bias_hh = b_hh;
                sa.x1 = lin; sa.x1_bstride = T;
                sa.t0 = 0; sa.steps = T;
                if (split_r1) { sa.xg = xg; sa.xg_bstride = (long long)T * GH; }      // delta_hh of every step
                sa.dh_in = dhTl;
                sa.dc_in = dcTl;
                sa.dh_out = sdh; sa.dc_out = sdc;
                if (launch_plan(sa)) return 1;
                if (split_r1) {
                    // hh core gradients: dense accumulation dW_hh^T = H_prev^T delta over rows (h_{t-1}, delta_t)
                    auto hh_dw1 = [&](const float *xp, long long xbs, const float *dyp, long long rows, int rpb) -> int {
                        if (dense_dw(dvw, rows, rpb, xp, xbs, H, dyp, (long long)T * GH, GH, DH, hh_dense_calls > 0, false, ws))
                            return 1;
                        ++hh_dense_calls;
                        return 0;
                    };
                    if (T > 1 && hh_dw1(lout, (long long)T * H, xg + GH, B * (T - 1), T - 1)) return 1;
                    if (h0l && hh_dw1(h0l, H, xg, B, 1)) return 1;
                }
            } else {
                sa.bias_hh = lstm ? nullptr : b_hh;
                const int nchunks = (T + lo.Tc - 1) / lo.Tc;
                for (int ci = nchunks - 1; ci >= 0; --ci) {
                    const int t0 = ci * lo.Tc;
                    const int tc = (T - t0 < lo.Tc) ? T - t0 : lo.Tc;
                    const bool last = (t0 + tc == T);
                    // the kept-gates kernels take the gate activations from the forward pass and only WRITE delta_ih
                    // into xg: recomputing the ih projection of the chunk would be wasted work
                    if (!br.kept && project(t0, tc)) return 1;
                    sa.t0 = t0; sa.steps = tc;
                    sa.xg = xg; sa.xg_bstride = (long long)tc * GH;
                    sa.dh_in = last ? dhTl : sdh;
                    sa.dc_in = last ? dcTl : sdc;
                    sa.dh_out = sdh; sa.dc_out = sdc;
                    if (launch_plan(sa)) return 1;
                    // bwd_overlap: fork only when this layer's BPTT grid leaves >= 24 SMs idle
                    const int idle_sms = dv.sms - sgrid;
                    if (side && l > 0 && nchunks == 1 && dense && dlin && idle_sms >= 24) {
                        // overlap: dX (the next layer's input) first, then everything that only produces parameter gradients
                        // moves to the side stream, planned for the SMs the next BPTT kernel leaves idle
                        if (project_dx(t0, tc)) return 1;
                        dx_done = true;
                        CU_CHECK(cudaEventRecord(side->fork, st));
                        CU_CHECK(cudaStreamWaitEvent(side->s, side->fork, 0));
                        ws = side->s;
                        join.used = true;
                        dvw.sms = idle_sms;
                    }
                    if (split) {
                        // hh core gradients over rows (h_{t-1}, delta_t) of this chunk: dense accumulation of
                        // dW_hh^T = H_prev^T delta (projected onto the cores after the last chunk), or a batched
                        // TT-matvec backward (second chain pass) when the dense order is disabled / does not fit
                        auto hh_dw = [&](const float *xp, long long xbs, const float *dyp, long long rows, int rpb) {
                            if (dense_hh) {
                                if (dense_dw(dvw, rows, rpb, xp, xbs, H, dyp, (long long)tc * GH, GH, DH, hh_dense_calls > 0,
                                             false, ws))
                                    return 1;
                                ++hh_dense_calls;
                                return 0;
                            }
                            return launch_ttlinear_bwd(lp.hh, dvw, rows, rpb, xp, xbs, params + lp.off_hh_cores, dyp,
                                                       (long long)tc * GH, nullptr, 0, part_hh, lo.nslots,
                                                       ss + lo.b_spill, 0, ws, &hh_used, &d->hh[l]);
                        };
                        if (t0 > 0) {
                            if (hh_dw(lout + (long long)(t0 - 1) * H, (long long)T * H, xg, B * tc, tc)) return 1;
                        } else {
                            if (tc > 1 && hh_dw(lout, (long long)T * H, xg + GH, B * (tc - 1), tc - 1)) return 1;
                            if (h0l && hh_dw(h0l, H, xg, B, 1)) return 1;
                        }
                    }
                    if (project_bwd(t0, tc, &ih_used)) return 1;
                }
                if (project_finish(&ih_used)) return 1;
                if (dense_hh && hh_dense_calls > 0) {
                    // dense dW_hh^T -> TT cores: H-row TT-matvec backward with the identity as input
                    if (launch_ttlinear_bwd(lp.hh, dvw, H, H, DH.eye, 0, params + lp.off_hh_cores, DH.dwt, 0, nullptr, 0,
                                            part_hh, lo.nslots, ss + lo.b_spill, 0, ws, &hh_used, &d->hh[l]))
                        return 1;
                }
            }
            // fold the per-CTA slots into the gradient blob
            const long long cf = lp.hh.core_floats;
            if (split_r1) {
                // part_hh holds the kernel's slots (biases, W_ih column) and is reused for the projection of the dense
                // dW_hh^T onto the cores after those have been folded
                if (d->has_bias) {
                    if (reduce_partials(part_hh, sgrid, slot, cf, GH, d_params + lp.off_hh_bias, ws)) return 1;
                    if (reduce_partials(part_hh, sgrid, slot, cf + 2 * GH, GH, d_params + lp.off_ih_bias, ws)) return 1;
                }
                if (reduce_partials(part_hh, sgrid, slot, cf + GH, GH, aux_g, ws)) return 1;
                CU_CHECK(cudaMemsetAsync(part_hh, 0, (size_t)hhw_slot * lo.nslots * 4, ws));
                if (hh_dense_calls > 0 &&
                    launch_ttlinear_bwd(lp.hh, dvw, H, H, DH.eye, 0, params + lp.off_hh_cores, DH.dwt, 0, nullptr, 0, part_hh,
                                        lo.nslots, ss + lo.b_spill, 0, ws, &hh_used, &d->hh[l]))
                    return 1;
                if (hh_used > 0) {
                    if (reduce_partials(part_hh, hh_used, hhw_slot, 0, (int)cf, d_params + lp.off_hh_cores, ws)) return 1;
                } else {
                    CU_CHECK(cudaMemsetAsync(d_params + lp.off_hh_cores, 0, (size_t)cf * 4, ws));      // T == 1 without h0
                }
                if (launch_ttlinear_bwd(lp.ih, dvw, 1, 1, one, 0, params + lp.off_ih_cores, aux_g, 0, nullptr, 0, part_ih,
                                        lo.nslots, ss + lo.b_spill, 0, ws, &ih_used))
                    return 1;
                if (reduce_partials(part_ih, ih_used, ih_slot, 0, lp.ih.core_floats, d_params + lp.off_ih_cores, ws)) return 1;
            } else if (split) {
                if (reduce_partials(part_hh, hh_used, hhw_slot, 0, (int)cf, d_params + lp.off_hh_cores, ws)) return 1;
            } else if (reduce_partials(part_hh, sgrid, slot, 0, (int)cf, d_params + lp.off_hh_cores, ws)) {
                return 1;
            }
            if (split_r1) {
                // everything was folded above
            } else if (mode == tts::MODE_RANK1) {
                if (d->has_bias) {
                    if (reduce_partials(part_hh, sgrid, slot, cf, GH, d_params + lp.off_hh_bias, ws)) return 1;
                    if (reduce_partials(part_hh, sgrid, slot, cf + 2 * GH, GH, d_params + lp.off_ih_bias, ws)) return 1;
                }
                // gradient of the dense W_ih column -> TT cores of W_ih (one-row TT-matvec backward)
                if (reduce_partials(part_hh, sgrid, slot, cf + GH, GH, aux_g, ws)) return 1;
                if (launch_ttlinear_bwd(lp.ih, dvw, 1, 1, one, 0, params + lp.off_ih_cores, aux_g, 0, nullptr, 0, part_ih,
                                        lo.nslots, ss + lo.b_spill, 0, ws, &ih_used))
                    return 1;
                if (reduce_partials(part_ih, ih_used, ih_slot, 0, lp.ih.core_floats, d_params + lp.off_ih_cores, ws)) return 1;
            } else {
                if (reduce_partials(part_ih, ih_used, ih_slot, 0, lp.ih.core_floats, d_params + lp.off_ih_cores, ws)) return 1;
                if (d->has_bias) {
                    if (dense) {
                        if (axpy1(D.dbias, d_params + lp.off_ih_bias, GH, 0, ws)) return 1;
                    } else if (reduce_partials(part_ih, ih_used, ih_slot, lp.ih.core_floats, GH, d_params + lp.off_ih_bias, ws)) {
                        return 1;
                    }
                    if (lstm) {
                        if (axpy1(d_params + lp.off_ih_bias, d_params + lp.off_hh_bias, GH, 0, ws)) return 1;
                    } else {
                        if (reduce_partials(part_hh, sgrid, slot, cf, GH, d_params + lp.off_hh_bias, ws)) return 1;
                    }
                }
            }
            if (ws != st) {                                   // the set stays busy until the side stream has passed this point
                CU_CHECK(cudaEventRecord(side->done[set], ws));
                set_busy[set] = true;
            }
            if (d_h0 && axpy1(sdh, sm.init(d_h0, l), lo.BH, !sm.stride && l != L - 1, st)) return 1;
            if (lstm && d_c0 && axpy1(sdc, sm.init(d_c0, l, true), lo.BH, !sm.stride && l != L - 1, st)) return 1;
            continue;
        }

        if (rp.P) {
            // projected LSTM: k_rnn_bwd_proj runs the projection chain forward and backward inside every BPTT step; the
            // per-CTA slots hold the hh core gradients, then the hr core gradients
            RnnBwdProjArgs a;
            memset(&a, 0, sizeof a);
            BwdProjCfg cfg;
            if (plan_bwd_proj(lp.hh, lp.hr, H, W, dv, B, &cfg)) return 1;
            a.p = cfg.p;
            a.q = cfg.q;
            const int R = cfg.R;
            a.R = R;
            a.spill = cfg.spill > 0 ? ss + lo.b_spill : nullptr;
            fill_tiles(cfg.p, R, a.tile, a.tile_bd, a.mg);
            fill_tiles(cfg.q, R, a.tile_q, a.tile_bd_q, a.mg_q);
            a.H = H; a.P = W; a.B = B; a.T = T;
            a.cores = params + lp.off_hh_cores;
            a.cores_q = params + lp.off_hr_cores;
            a.hs = lout; a.cs = lcs; a.h0 = h0l; a.c0 = c0l; a.dhs = dhs;
            int grid = 0;
            if (grid_for(k_rnn_bwd_proj, cfg.smem, (B + R - 1) / R, dv, &grid)) return 1;
            if (grid > lo.nslots) grid = lo.nslots;
            const long long hh_slot = lp.hh.core_floats + lp.hr.core_floats;
            const long long ih_slot = lp.ih.core_floats + GH;
            CU_CHECK(cudaMemsetAsync(part_hh, 0, (size_t)hh_slot * grid * 4, st));
            CU_CHECK(cudaMemsetAsync(part_ih, 0, (size_t)ih_slot * lo.nslots * 4, st));
            a.partial = part_hh;
            int ih_slots_used = 0;
            const int nchunks = (T + lo.Tc - 1) / lo.Tc;
            for (int ci = nchunks - 1; ci >= 0; --ci) {
                const int t0 = ci * lo.Tc;
                const int tc = (T - t0 < lo.Tc) ? T - t0 : lo.Tc;
                const bool last = (t0 + tc == T);
                if (project(t0, tc)) return 1;
                a.t0 = t0; a.steps = tc;
                a.xg = xg; a.xg_bstride = (long long)tc * GH;
                a.dh_in = last ? dhTl : sdh;
                a.dc_in = last ? dcTl : sdc;
                a.dh_out = sdh; a.dc_out = sdc;
                {
                    KernelTimer tm(TTRNN_K_RNN_BWD, st, R, grid, B, tc);
                    k_rnn_bwd_proj<<<grid, TT_NTHREADS, cfg.smem, st>>>(a);
                }
                ++g_launches;
                CU_CHECK(cudaGetLastError());
                if (project_bwd(t0, tc, &ih_slots_used)) return 1;
            }
            if (project_finish(&ih_slots_used)) return 1;
            if (reduce_partials(part_hh, grid, hh_slot, 0, lp.hh.core_floats, d_params + lp.off_hh_cores, st)) return 1;
            if (reduce_partials(part_hh, grid, hh_slot, lp.hh.core_floats, lp.hr.core_floats, d_params + lp.off_hr_cores, st))
                return 1;
            if (reduce_partials(part_ih, ih_slots_used, ih_slot, 0, lp.ih.core_floats, d_params + lp.off_ih_cores, st)) return 1;
            if (d->has_bias) {
                if (dense) {
                    if (axpy1(D.dbias, d_params + lp.off_ih_bias, GH, 0, st)) return 1;
                } else if (reduce_partials(part_ih, ih_slots_used, ih_slot, lp.ih.core_floats, GH, d_params + lp.off_ih_bias, st)) {
                    return 1;
                }
                if (axpy1(d_params + lp.off_ih_bias, d_params + lp.off_hh_bias, GH, 0, st)) return 1;
            }
            if (d_h0 && axpy1(sdh, sm.init(d_h0, l), lo.BW, !sm.stride && l != L - 1, st)) return 1;
            if (d_c0 && axpy1(sdc, sm.init(d_c0, l, true), lo.BH, !sm.stride && l != L - 1, st)) return 1;
            continue;
        }

        RnnBwdArgs a;
        memset(&a, 0, sizeof a);
        BwdCfg cfg;
        if (plan_bwd(lp.hh, [&](int r) { return smem_rnn_bwd_fixed(lp.hh, r, H, G); }, dv, B, &cfg, "hh backward")) return 1;
        a.p = cfg.p;
        const int R = cfg.R;
        a.R = R;
        a.spill = cfg.spill > 0 ? ss + lo.b_spill : nullptr;
        fill_tiles(cfg.p, R, a.tile, a.tile_bd, a.mg);
        a.cell = d->cell; a.H = H; a.G = G; a.B = B; a.T = T;
        a.cores = params + lp.off_hh_cores;
        a.bias_hh = lstm ? nullptr : b_hh;
        a.hs = lout; a.cs = lcs; a.h0 = h0l; a.c0 = c0l; a.dhs = dhs;
        if (logging) {
            a.dh_log = t_log.dh + (long long)l * t_log.layer_stride;
            a.dc_log = (lstm && t_log.dc) ? t_log.dc + (long long)l * t_log.layer_stride : nullptr;
        }
        const size_t smem = cfg.smem;
        int grid = 0;
        if (grid_for(k_rnn_bwd, smem, (B + R - 1) / R, dv, &grid)) return 1;
        if (grid > lo.nslots) grid = lo.nslots;
        const long long hh_slot = lp.hh.core_floats + GH;
        const long long ih_slot = lp.ih.core_floats + GH;
        CU_CHECK(cudaMemsetAsync(part_hh, 0, (size_t)hh_slot * grid * 4, st));
        CU_CHECK(cudaMemsetAsync(part_ih, 0, (size_t)ih_slot * lo.nslots * 4, st));
        a.partial = part_hh;
        int ih_slots_used = 0;

        const int nchunks = (T + lo.Tc - 1) / lo.Tc;
        for (int ci = nchunks - 1; ci >= 0; --ci) {
            const int t0 = ci * lo.Tc;
            const int tc = (T - t0 < lo.Tc) ? T - t0 : lo.Tc;
            const bool last = (t0 + tc == T);
            // (1) recompute the ih projection of the chunk
            if (project(t0, tc)) return 1;
            // (2) reverse-time recurrence: xg <- delta_ih, hh core grads, dh/dc carried across chunks
            a.t0 = t0; a.steps = tc;
            a.xg = xg; a.xg_bstride = (long long)tc * GH;
            a.dh_in = last ? dhTl : sdh;
            a.dc_in = last ? dcTl : sdc;
            a.dh_out = sdh; a.dc_out = sdc;
            {
                KernelTimer tm(TTRNN_K_RNN_BWD, st, R, grid, B, tc);
                k_rnn_bwd<<<grid, TT_NTHREADS, smem, st>>>(a);
            }
            ++g_launches;
            CU_CHECK(cudaGetLastError());
            // (3) ih backward over the chunk: core grads, bias grad, gradient wrt the layer input
            if (project_bwd(t0, tc, &ih_slots_used)) return 1;
        }
        if (project_finish(&ih_slots_used)) return 1;
        // (4) fold the per-CTA partials into the gradient blob
        if (reduce_partials(part_hh, grid, hh_slot, 0, lp.hh.core_floats, d_params + lp.off_hh_cores, st)) return 1;
        if (reduce_partials(part_ih, ih_slots_used, ih_slot, 0, lp.ih.core_floats, d_params + lp.off_ih_cores, st)) return 1;
        if (d->has_bias) {
            if (dense) {
                if (axpy1(D.dbias, d_params + lp.off_ih_bias, GH, 0, st)) return 1;
            } else if (reduce_partials(part_ih, ih_slots_used, ih_slot, lp.ih.core_floats, GH, d_params + lp.off_ih_bias, st)) {
                return 1;
            }
            if (lstm) {
                if (axpy1(d_params + lp.off_ih_bias, d_params + lp.off_hh_bias, GH, 0, st)) return 1;
            } else {
                if (reduce_partials(part_hh, grid, hh_slot, lp.hh.core_floats, GH, d_params + lp.off_hh_bias, st)) return 1;
            }
        }
        // (5) gradient wrt the initial state: this layer's own block, or the sum over layers when the state is shared
        if (d_h0 && axpy1(sdh, sm.init(d_h0, l), lo.BH, !sm.stride && l != L - 1, st)) return 1;
        if (lstm && d_c0 && axpy1(sdc, sm.init(d_c0, l, true), lo.BH, !sm.stride && l != L - 1, st)) return 1;
    }
    return 0;
}

// per-layer state buffers (TTRNN_WS_LAYER_STATES in the plan) are strided by the full batch's B * H, so that a row group
// reaches layer l's rows from a pointer moved to its first row
static StateMap state_map(const ttrnn_rnn_desc *d_full, const ttrnn_rnn_workspace *ws, const ttrnn_rnn_proj *pj) {
    StateMap sm;
    if (ws->plan[kPlanLayerStates]) {
        sm.cstride = (long long)d_full->batch * d_full->hidden_size;
        sm.stride = pj ? (long long)d_full->batch * pj->proj_size : sm.cstride;
    }
    return sm;
}

// the projection of an entry point: proj_given = the call is a _proj entry point (which requires pj and a plan sized
// with TTRNN_WS_PROJ); every other entry point refuses such a plan
static int proj_call(const char *who, const ttrnn_rnn_desc *d_in, const ttrnn_rnn_workspace *ws, bool proj_given,
                     const ttrnn_rnn_proj *pj) {
    if (!proj_given) {
        if (ws->plan[kPlanProj])
            return fail("%s: the plan was sized with TTRNN_WS_PROJ; run it with the _proj entry points", who);
        return 0;
    }
    if (!ws->plan[kPlanProj]) return fail("%s: the plan was not sized with TTRNN_WS_PROJ (ttrnn_rnn_workspace_bytes_proj)", who);
    if (!pj) return fail("%s: pj must be non-null", who);
    if (d_in->cell != TTRNN_CELL_LSTM) return fail("%s: a projection needs an LSTM descriptor", who);
    return 0;
}

// ---- public entry points: one call of the single-group path per row group ---------------------------------------
// Group 0 runs on the caller's stream, group 1 on the group stream, forked from the caller's stream at entry (so that it
// waits for whatever produced the inputs, not for group 0) and joined at exit.  While per-kernel event timing is on
// (ttrnn_kernel_timing, bench only) the groups run back to back on the caller's stream: events around launches that
// share the SMs with another stream's kernels would not measure those kernels.
struct GroupSlices {
    int n = 1;
    long long row0[kMaxGroups] = {0, 0};
    ttrnn_rnn_desc d[kMaxGroups];
    ttrnn_rnn_workspace w[kMaxGroups];
    int64_t sv_off[kMaxGroups] = {0, 0}, f_off[kMaxGroups] = {0, 0}, b_off[kMaxGroups] = {0, 0}, dp_off[kMaxGroups] = {0, 0};
};
static int group_slices(const ttrnn_rnn_desc *d_in, const ttrnn_rnn_workspace *ws, GroupSlices *gs, const char *who) {
    const long long ng = ws->plan[kPlanGroups], rows0 = ws->plan[kPlanRows0];
    if (!d_in) return fail("null descriptor");
    if (ng != 2 || rows0 <= 0 || rows0 >= d_in->batch)
        return fail("%s: workspace struct does not belong to this descriptor (row groups %lld, %lld of %lld rows)", who, ng, rows0,
                    (long long)d_in->batch);
    const int64_t pf = ttrnn_rnn_param_count(d_in);
    if (pf < 0) return 1;
    gs->n = 2;
    int64_t sv = 0, f = 0, b = 0;
    for (int g = 0; g < 2; ++g) {
        gs->row0[g] = g ? rows0 : 0;
        gs->d[g] = *d_in;
        gs->d[g].batch = g ? d_in->batch - rows0 : rows0;
        if (workspace_one(&gs->d[g], &gs->w[g], ws->plan[kPlanDropout] != 0)) return 1;
        memcpy(gs->w[g].plan, ws->plan, sizeof ws->plan);
        gs->sv_off[g] = sv; sv += a256(gs->w[g].saved_bytes);
        gs->f_off[g] = f;   f += a256(gs->w[g].fwd_scratch_bytes);
        gs->b_off[g] = b;   b += a256(gs->w[g].bwd_scratch_bytes);
        if (g > 0) { gs->dp_off[g] = b; b += a256(pf * 4); }
    }
    if (sv != ws->saved_bytes || f != ws->fwd_scratch_bytes || b != ws->bwd_scratch_bytes)
        return fail("%s: workspace struct does not belong to this descriptor (group sizes %lld / %lld / %lld bytes vs %lld / %lld / %lld)",
                    who, (long long)sv, (long long)f, (long long)b, (long long)ws->saved_bytes, (long long)ws->fwd_scratch_bytes,
                    (long long)ws->bwd_scratch_bytes);
    return 0;
}

// the mask of a dropout entry point: nullptr when there is none to apply (no dp, or a one-layer stack).  `who` names the
// entry point in errors; dp_given: the call is a dropout entry point (which requires dp)
static int drop_call(const char *who, const ttrnn_rnn_desc *d_in, const ttrnn_rnn_workspace *ws, bool dp_given,
                     const ttrnn_dropout *dp, DropCall *dc, const DropCall **out) {
    *out = nullptr;
    if (!dp_given) {
        if (ws->plan[kPlanDropout])
            return fail("%s: the plan was sized with TTRNN_WS_DROPOUT; run it with the _dropout entry points", who);
        return 0;
    }
    if (!dp) return fail("%s: dp must be non-null", who);
    if (!(dp->p >= 0.f && dp->p <= 1.f)) return fail("%s: dropout p must be in [0, 1], got %g", who, (double)dp->p);
    if (dp->p > 0.f && !ws->plan[kPlanDropout])
        return fail("%s: dropout p > 0 needs a plan sized with TTRNN_WS_DROPOUT", who);
    if (d_in->num_layers < 2 || !ws->plan[kPlanDropout]) return 0;       // nothing between layers / p = 0 without buffers
    dc->p = dp->p; dc->seed = dp->seed; dc->offset = dp->offset; dc->row0 = 0;
    *out = dc;
    return 0;
}

static int rnn_forward_entry(const char *who, const ttrnn_rnn_desc *d_in, const ttrnn_rnn_workspace *ws, const float *x,
                             const float *h0, const float *c0, const float *params, float *out, float *hT, float *cT,
                             void *saved, void *scratch, void *stream, bool dp_given, const ttrnn_dropout *dp,
                             bool proj_given = false, const ttrnn_rnn_proj *pj = nullptr) {
    if (!ws || !plan_load(ws->plan, &t_opt))
        return fail("%s: `ws` must be the struct filled by ttrnn_rnn_workspace_bytes() for this descriptor", who);
    if (!d_in) return fail("null descriptor");
    if (proj_call(who, d_in, ws, proj_given, pj)) return 1;
    DropCall dcs;
    const DropCall *dc = nullptr;
    if (drop_call(who, d_in, ws, dp_given, dp, &dcs, &dc)) return 1;
    const StateMap sm = state_map(d_in, ws, pj);
    if (ws->plan[kPlanGroups] <= 1)
        return forward_one(d_in, ws, sm, x, h0, c0, params, out, hT, cT, saved, scratch, stream, dc, pj);
    if (!x || !params || !out || !scratch) return fail("x, params, out and scratch must be non-null");
    GroupSlices gs;
    if (group_slices(d_in, ws, &gs, "ttrnn_rnn_forward")) return 1;
    GroupCtx *gc = group_ctx();
    if (!gc) return fail("ttrnn_rnn_forward: cannot create the row-group stream");
    cudaStream_t st = (cudaStream_t)stream;
    const bool serial = g_timing.load() != 0;
    if (!serial) {
        CU_CHECK(cudaEventRecord(gc->fork, st));
        CU_CHECK(cudaStreamWaitEvent(gc->s, gc->fork, 0));
    }
    const long long T = d_in->seq_len, I = d_in->input_size, H = d_in->hidden_size;
    int rc = 0;
    for (int g = 0; g < gs.n && !rc; ++g) {
        const long long r0 = gs.row0[g];
        t_group = g;
        if (dc) dcs.row0 = r0;                  // the mask is indexed by global rows
        rc = forward_one(&gs.d[g], &gs.w[g], sm, x + r0 * T * I, h0 ? h0 + r0 * H : nullptr, c0 ? c0 + r0 * H : nullptr, params,
                         out + r0 * T * H, hT ? hT + r0 * H : nullptr, cT ? cT + r0 * H : nullptr,
                         saved ? (char *)saved + gs.sv_off[g] : nullptr, (char *)scratch + gs.f_off[g],
                         (g == 0 || serial) ? (void *)st : (void *)gc->s, dc, nullptr);
    }
    t_group = 0;
    if (!serial) {       // also on the error path: the caller's stream must not run ahead of the group stream
        cudaEventRecord(gc->join, gc->s);
        cudaStreamWaitEvent(st, gc->join, 0);
    }
    return rc;
}

int ttrnn_rnn_forward(const ttrnn_rnn_desc *d_in, const ttrnn_rnn_workspace *ws, const float *x, const float *h0,
                      const float *c0, const float *params, float *out, float *hT, float *cT, void *saved, void *scratch,
                      void *stream) {
    return rnn_forward_entry("ttrnn_rnn_forward", d_in, ws, x, h0, c0, params, out, hT, cT, saved, scratch, stream, false,
                             nullptr);
}

int ttrnn_rnn_forward_dropout(const ttrnn_rnn_desc *d_in, const ttrnn_rnn_workspace *ws, const float *x, const float *h0,
                              const float *c0, const float *params, float *out, float *hT, float *cT, void *saved,
                              void *scratch, void *stream, const ttrnn_dropout *dp) {
    return rnn_forward_entry("ttrnn_rnn_forward_dropout", d_in, ws, x, h0, c0, params, out, hT, cT, saved, scratch, stream,
                             true, dp);
}

static int rnn_backward_entry(const char *who, const ttrnn_rnn_desc *d_in, const ttrnn_rnn_workspace *ws, const float *x,
                              const float *h0, const float *c0, const float *params, const float *out, const void *saved,
                              const float *d_out, const float *d_hT, const float *d_cT, float *d_params, float *d_x,
                              float *d_h0, float *d_c0, void *scratch, void *stream, bool dp_given, const ttrnn_dropout *dp,
                              bool proj_given = false, const ttrnn_rnn_proj *pj = nullptr) {
    if (!ws || !plan_load(ws->plan, &t_opt))
        return fail("%s: `ws` must be the struct the matching forward ran with", who);
    if (!d_in) return fail("null descriptor");
    if (proj_call(who, d_in, ws, proj_given, pj)) return 1;
    DropCall dcs;
    const DropCall *dc = nullptr;
    if (drop_call(who, d_in, ws, dp_given, dp, &dcs, &dc)) return 1;
    const StateMap sm = state_map(d_in, ws, pj);
    if (ws->plan[kPlanGroups] <= 1)
        return backward_one(d_in, ws, sm, x, h0, c0, params, out, saved, d_out, d_hT, d_cT, d_params, d_x, d_h0, d_c0, scratch,
                            stream, dc, pj);
    if (!x || !params || !out || !scratch || !d_params) return fail("x, params, out, scratch, d_params must be non-null");
    GroupSlices gs;
    if (group_slices(d_in, ws, &gs, "ttrnn_rnn_backward")) return 1;
    GroupCtx *gc = group_ctx();
    if (!gc) return fail("ttrnn_rnn_backward: cannot create the row-group stream");
    cudaStream_t st = (cudaStream_t)stream;
    const bool serial = g_timing.load() != 0;
    if (!serial) {
        CU_CHECK(cudaEventRecord(gc->fork, st));
        CU_CHECK(cudaStreamWaitEvent(gc->s, gc->fork, 0));
    }
    const long long T = d_in->seq_len, I = d_in->input_size, H = d_in->hidden_size;
    const int64_t pf = ttrnn_rnn_param_count(d_in);
    int rc = 0;
    for (int g = 0; g < gs.n && !rc; ++g) {
        const long long r0 = gs.row0[g];
        float *dp = g == 0 ? d_params : (float *)((char *)scratch + gs.dp_off[g]);
        t_group = g;
        if (dc) dcs.row0 = r0;
        rc = backward_one(&gs.d[g], &gs.w[g], sm, x + r0 * T * I, h0 ? h0 + r0 * H : nullptr, c0 ? c0 + r0 * H : nullptr, params,
                          out + r0 * T * H, saved ? (const char *)saved + gs.sv_off[g] : nullptr,
                          d_out ? d_out + r0 * T * H : nullptr, d_hT ? d_hT + r0 * H : nullptr, d_cT ? d_cT + r0 * H : nullptr, dp,
                          d_x ? d_x + r0 * T * I : nullptr, d_h0 ? d_h0 + r0 * H : nullptr, d_c0 ? d_c0 + r0 * H : nullptr,
                          (char *)scratch + gs.b_off[g], (g == 0 || serial) ? (void *)st : (void *)gc->s, dc, nullptr);
    }
    t_group = 0;
    if (!serial) {
        cudaEventRecord(gc->join, gc->s);
        cudaStreamWaitEvent(st, gc->join, 0);
    }
    if (rc) return rc;
    // parameter gradients: sum of the groups' blobs
    for (int g = 1; g < gs.n; ++g)
        if (axpy1((const float *)((char *)scratch + gs.dp_off[g]), d_params, pf, 1, st)) return 1;
    return 0;
}

int ttrnn_rnn_backward(const ttrnn_rnn_desc *d_in, const ttrnn_rnn_workspace *ws, const float *x, const float *h0,
                       const float *c0, const float *params, const float *out, const void *saved, const float *d_out,
                       const float *d_hT, const float *d_cT, float *d_params, float *d_x, float *d_h0, float *d_c0,
                       void *scratch, void *stream) {
    return rnn_backward_entry("ttrnn_rnn_backward", d_in, ws, x, h0, c0, params, out, saved, d_out, d_hT, d_cT, d_params, d_x,
                              d_h0, d_c0, scratch, stream, false, nullptr);
}

int ttrnn_rnn_backward_dropout(const ttrnn_rnn_desc *d_in, const ttrnn_rnn_workspace *ws, const float *x, const float *h0,
                               const float *c0, const float *params, const float *out, const void *saved, const float *d_out,
                               const float *d_hT, const float *d_cT, float *d_params, float *d_x, float *d_h0, float *d_c0,
                               void *scratch, void *stream, const ttrnn_dropout *dp) {
    return rnn_backward_entry("ttrnn_rnn_backward_dropout", d_in, ws, x, h0, c0, params, out, saved, d_out, d_hT, d_cT,
                              d_params, d_x, d_h0, d_c0, scratch, stream, true, dp);
}

int ttrnn_rnn_forward_proj(const ttrnn_rnn_desc *d_in, const ttrnn_rnn_workspace *ws, const float *x, const float *h0,
                           const float *c0, const float *params, float *out, float *hT, float *cT, void *saved, void *scratch,
                           void *stream, const ttrnn_rnn_proj *pj, const ttrnn_dropout *dp) {
    return rnn_forward_entry("ttrnn_rnn_forward_proj", d_in, ws, x, h0, c0, params, out, hT, cT, saved, scratch, stream,
                             dp != nullptr, dp, true, pj);
}

int ttrnn_rnn_backward_proj(const ttrnn_rnn_desc *d_in, const ttrnn_rnn_workspace *ws, const float *x, const float *h0,
                            const float *c0, const float *params, const float *out, const void *saved, const float *d_out,
                            const float *d_hT, const float *d_cT, float *d_params, float *d_x, float *d_h0, float *d_c0,
                            void *scratch, void *stream, const ttrnn_rnn_proj *pj, const ttrnn_dropout *dp) {
    return rnn_backward_entry("ttrnn_rnn_backward_proj", d_in, ws, x, h0, c0, params, out, saved, d_out, d_hT, d_cT, d_params,
                              d_x, d_h0, d_c0, scratch, stream, dp != nullptr, dp, true, pj);
}

int ttrnn_dropout_apply(int64_t B, int32_t T, int32_t F, int64_t row0, int32_t boundary, int32_t backward,
                        const ttrnn_dropout *dp, const float *x, float *y, float *y_rev, void *stream) {
    if (B < 1 || T < 1 || F < 1 || row0 < 0) return fail("ttrnn_dropout_apply: B, T, F must be >= 1 and row0 >= 0 (got %lld, %d, %d, %lld)",
                                                         (long long)B, T, F, (long long)row0);
    if (boundary < 0 || boundary >= TTRNN_MAX_LAYERS) return fail("ttrnn_dropout_apply: boundary %d out of range", boundary);
    if (!dp) return fail("ttrnn_dropout_apply: dp must be non-null");
    if (!(dp->p >= 0.f && dp->p <= 1.f)) return fail("ttrnn_dropout_apply: dropout p must be in [0, 1], got %g", (double)dp->p);
    if (!x || !y) return fail("ttrnn_dropout_apply: x and y must be non-null");
    if (y_rev && (y_rev == y || y_rev == x)) return fail("ttrnn_dropout_apply: y_rev must not alias x or y");
    DevInfo dv;
    if (get_dev(&dv)) return 1;
    DropCall dc;
    dc.p = dp->p; dc.seed = dp->seed; dc.offset = dp->offset; dc.row0 = row0;
    if (backward) return launch_dropout(dv, B, T, F, dc, row0, boundary, x, y_rev, y, nullptr, (cudaStream_t)stream);
    return launch_dropout(dv, B, T, F, dc, row0, boundary, x, nullptr, y, y_rev, (cudaStream_t)stream);
}

int ttrnn_rnn_backward_logged(const ttrnn_rnn_desc *d_in, const ttrnn_rnn_workspace *ws, const float *x, const float *h0,
                              const float *c0, const float *params, const float *out, const void *saved, const float *d_out,
                              const float *d_hT, const float *d_cT, float *d_params, float *d_x, float *d_h0, float *d_c0,
                              void *scratch, void *stream, float *dh_log, float *dc_log) {
    if (!d_in || !ws) return fail("null descriptor / workspace struct");
    if (!dh_log) return fail("ttrnn_rnn_backward_logged: dh_log must be non-null");
    if (ws->plan[kPlanDropout]) return fail("ttrnn_rnn_backward_logged: the plan was sized with TTRNN_WS_DROPOUT");
    if (ws->plan[kPlanProj]) return fail("ttrnn_rnn_backward_logged: the plan was sized with TTRNN_WS_PROJ");
    if (ws->plan[kPlanGroups] > 1)
        return fail("ttrnn_rnn_backward_logged needs a whole-batch plan: size the call with "
                    "ttrnn_rnn_workspace_bytes_ex(desc, TTRNN_WS_WHOLE_BATCH, ws)");
    t_log.dh = dh_log;
    t_log.dc = dc_log;
    t_log.layer_stride = (long long)d_in->batch * d_in->seq_len * d_in->hidden_size;
    const int rc = ttrnn_rnn_backward(d_in, ws, x, h0, c0, params, out, saved, d_out, d_hT, d_cT, d_params, d_x, d_h0, d_c0,
                                      scratch, stream);
    t_log = StepLog();
    return rc;
}

int ttrnn_rnn_saved_layout(const ttrnn_rnn_desc *d_in, const ttrnn_rnn_workspace *ws, int32_t layer, int64_t *hs_off,
                           int64_t *cs_off) {
    if (!ws || !plan_load(ws->plan, &t_opt)) return fail("ttrnn_rnn_saved_layout: `ws` must come from ttrnn_rnn_workspace_bytes()");
    if (ws->plan[kPlanGroups] > 1) return fail("ttrnn_rnn_saved_layout needs a whole-batch plan (TTRNN_WS_WHOLE_BATCH)");
    if (ws->plan[kPlanProj]) return fail("ttrnn_rnn_saved_layout: the plan was sized with TTRNN_WS_PROJ");
    if (!hs_off || !cs_off) return fail("hs_off and cs_off must be non-null");
    DevInfo dv;
    CallPlan cp;
    if (get_dev(&dv) || plan_call(d_in, dv, &cp, ws->plan[kPlanDropout] != 0)) return 1;
    if (layer < 0 || layer >= d_in->num_layers) return fail("layer %d out of range", layer);
    *hs_off = (layer == d_in->num_layers - 1) ? -1 : cp.lo.sv_hs + (long long)layer * cp.lo.BTH;
    *cs_off = (d_in->cell == TTRNN_CELL_LSTM) ? cp.lo.sv_cs + (long long)layer * cp.lo.BTH : -1;
    return 0;
}

int ttrnn_step_norms(const float *v, int64_t B, int32_t T, int32_t H, float *out, void *stream) {
    if (!v || !out || B < 1 || T < 1 || H < 1) return fail("ttrnn_step_norms: bad arguments");
    k_step_norms<<<(unsigned)T, 256, 0, (cudaStream_t)stream>>>(v, B, T, H, out);
    ++g_launches;
    CU_CHECK(cudaGetLastError());
    return 0;
}

// ---- bidirectional stacks: time-reversed moves around the one-layer calls (tt_bidir.cuh) ---------------------------

int ttrnn_time_reverse_add(int64_t B, int32_t T, int32_t F, const float *a, const float *r, float *y, void *stream) {
    if (B < 1 || T < 1 || F < 1) return fail("ttrnn_time_reverse_add: B, T and F must be >= 1 (got %lld, %d, %d)",
                                             (long long)B, T, F);
    if (!y) return fail("ttrnn_time_reverse_add: y is NULL");
    DevInfo dv;
    if (get_dev(&dv)) return 1;
    cudaStream_t st = (cudaStream_t)stream;
    if (F % 4 == 0 && aligned16(a) && aligned16(r) && aligned16(y)) {
        const long long n = B * (long long)T * (F / 4);
        bidir::k_reverse_add<4><<<bidir::grid_for(n, dv.sms), bidir::NT, 0, st>>>(a, r, y, n, T, F / 4);
    } else {
        const long long n = B * (long long)T * F;
        bidir::k_reverse_add<1><<<bidir::grid_for(n, dv.sms), bidir::NT, 0, st>>>(a, r, y, n, T, F);
    }
    ++g_launches;
    CU_CHECK(cudaGetLastError());
    return 0;
}

int ttrnn_bidir_join(int64_t B, int32_t T, int32_t H, int32_t backward, const float *p, const float *q, float *u,
                     float *v, void *stream) {
    if (B < 1 || T < 1 || H < 1) return fail("ttrnn_bidir_join: B, T and H must be >= 1 (got %lld, %d, %d)",
                                             (long long)B, T, H);
    if (!u || (backward && !v)) return fail("ttrnn_bidir_join: missing output");
    if (!backward && (!p || !q)) return fail("ttrnn_bidir_join: the forward needs both directions' outputs");
    DevInfo dv;
    if (get_dev(&dv)) return 1;
    cudaStream_t st = (cudaStream_t)stream;
    const bool vec = H % 4 == 0 && aligned16(p) && aligned16(q) && aligned16(u) && aligned16(v);
    const int V = vec ? 4 : 1;
    const long long n = B * (long long)T * (H / V) * (backward ? 1 : 2);
    const unsigned grid = bidir::grid_for(n, dv.sms);
    if (backward) {
        if (vec) bidir::k_join_bwd<4><<<grid, bidir::NT, 0, st>>>(p, q, u, v, n, T, H / 4);
        else bidir::k_join_bwd<1><<<grid, bidir::NT, 0, st>>>(p, q, u, v, n, T, H);
    } else {
        if (vec) bidir::k_join_fwd<4><<<grid, bidir::NT, 0, st>>>(p, q, u, v, n, T, H / 4);
        else bidir::k_join_fwd<1><<<grid, bidir::NT, 0, st>>>(p, q, u, v, n, T, H);
    }
    ++g_launches;
    CU_CHECK(cudaGetLastError());
    return 0;
}

// ---- stand-alone TTLinear -----------------------------------------------------------------------
int64_t ttrnn_ttlinear_param_count(const ttrnn_tt_shape *shape) {
    ChainPlan p;
    if (!shape || tt_build_plan(shape, &p)) { fail("malformed TT shape"); return -1; }
    return p.core_floats;
}

int64_t ttrnn_ttlinear_workspace_bytes(const ttrnn_tt_shape *shape, int64_t rows) {
    t_opt = snapshot_options();
    ChainPlan p;
    if (!shape || tt_build_plan(shape, &p)) { fail("malformed TT shape"); return -1; }
    DevInfo dv;
    if (get_dev(&dv)) return -1;
    BwdCfg c;
    if (plan_bwd(p, [&](int r) { return smem_ttlin_bwd_fixed(p, r); }, dv, rows > 0 ? rows : 1, &c, "TT matvec backward"))
        return -1;
    return (int64_t)(r4(p.core_floats + p.n_out) + r4(c.spill)) * dv.sms * kMaxSlotsPerSM * 4;
}

int ttrnn_ttlinear_forward(const ttrnn_tt_shape *shape, int64_t rows, const float *x, const float *cores,
                           const float *bias, float *y, void *scratch, void *stream) {
    (void)scratch;
    t_opt = snapshot_options();
    ChainPlan p;
    if (!shape || tt_build_plan(shape, &p)) return fail("malformed TT shape");
    if (rows < 1) return fail("rows must be >= 1");
    if (!x || !cores || !y) return fail("x, cores and y must be non-null");
    DevInfo dv;
    if (get_dev(&dv)) return 1;
    if (rows > 0x7fffffffLL) return fail("rows too large");
    return launch_ttlinear_fwd(p, dv, rows, (int)rows, x, 0, cores, bias, nullptr, y, 0, (cudaStream_t)stream, shape);
}

int ttrnn_ttlinear_backward(const ttrnn_tt_shape *shape, int64_t rows, const float *x, const float *cores,
                            const float *dy, float *d_x, float *d_cores, float *d_bias, void *scratch, void *stream) {
    t_opt = snapshot_options();
    ChainPlan p;
    if (!shape || tt_build_plan(shape, &p)) return fail("malformed TT shape");
    if (rows < 1 || rows > 0x7fffffffLL) return fail("rows out of range");
    if (!x || !cores || !dy || !d_cores || !scratch) return fail("x, cores, dy, d_cores, scratch must be non-null");
    DevInfo dv;
    if (get_dev(&dv)) return 1;
    cudaStream_t st = (cudaStream_t)stream;
    const int nslots = dv.sms * kMaxSlotsPerSM;
    const long long slot = p.core_floats + p.n_out;
    float *part = (float *)scratch;
    CU_CHECK(cudaMemsetAsync(part, 0, (size_t)slot * nslots * 4, st));
    int used = 0;
    float *spill = part + r4(slot) * nslots;
    if (launch_ttlinear_bwd(p, dv, rows, (int)rows, x, 0, cores, dy, 0, d_x, 0, part, nslots, spill,
                            d_bias != nullptr, st, &used, shape))
        return 1;
    if (reduce_partials(part, used, slot, 0, p.core_floats, d_cores, st)) return 1;
    if (d_bias && reduce_partials(part, used, slot, p.core_floats, p.n_out, d_bias, st)) return 1;
    return 0;
}

// ---- stand-alone cell step (cell-step mode: is_naive / log_grads) -------------------------------
static int cell_args_ok(int cell, int64_t B, int H) {
    if (cell != TTRNN_CELL_LSTM && cell != TTRNN_CELL_GRU) return fail("unknown cell kind %d", cell);
    if (B < 1 || H < 1) return fail("batch and hidden_size must be >= 1");
    return 0;
}

int ttrnn_cell_forward(int32_t cell, int64_t B, int32_t H, const float *a, const float *u, const float *h_prev,
                       const float *c_prev, float *h, float *c, void *stream) {
    if (cell_args_ok(cell, B, H)) return 1;
    const bool lstm = cell == TTRNN_CELL_LSTM;
    if (!a || !u || !h || (lstm ? (!c_prev || !c) : !h_prev)) return fail("ttrnn_cell_forward: null operand");
    DevInfo dv;
    if (get_dev(&dv)) return 1;
    CellStepArgs p;
    memset(&p, 0, sizeof p);
    p.B = B; p.H = H; p.a = a; p.u = u; p.h_prev = h_prev; p.c_prev = c_prev; p.h = h; p.c = c;
    long long blocks = (B * (long long)H + 255) / 256;
    if (blocks > (long long)dv.sms * 8) blocks = (long long)dv.sms * 8;
    if (lstm) k_cell_fwd<true><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(p);
    else k_cell_fwd<false><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(p);
    ++g_launches;
    CU_CHECK(cudaGetLastError());
    return 0;
}

int ttrnn_cell_backward(int32_t cell, int64_t B, int32_t H, const float *a, const float *u, const float *h_prev,
                        const float *c_prev, const float *dh, const float *dc, float *da, float *du,
                        float *dh_prev, float *dc_prev, float *dc_total, void *stream) {
    if (cell_args_ok(cell, B, H)) return 1;
    const bool lstm = cell == TTRNN_CELL_LSTM;
    if (!a || !u || !da || !du || !dh_prev || (lstm ? (!c_prev || !dc_prev) : !h_prev))
        return fail("ttrnn_cell_backward: null operand");
    DevInfo dv;
    if (get_dev(&dv)) return 1;
    CellStepArgs p;
    memset(&p, 0, sizeof p);
    p.B = B; p.H = H; p.a = a; p.u = u; p.h_prev = h_prev; p.c_prev = c_prev; p.dh = dh; p.dc = dc;
    p.da = da; p.du = du; p.dh_prev = dh_prev; p.dc_prev = dc_prev; p.dc_total = dc_total;
    long long blocks = (B * (long long)H + 255) / 256;
    if (blocks > (long long)dv.sms * 8) blocks = (long long)dv.sms * 8;
    if (lstm) k_cell_bwd<true><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(p);
    else k_cell_bwd<false><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(p);
    ++g_launches;
    CU_CHECK(cudaGetLastError());
    return 0;
}

// ---- dense LSTM / GRU baselines (SURVEY.md 8f-3) -----------------------------------------------------------------
namespace {
struct DenseLayerOff { long long w_ih, b_ih, w_hh, b_hh; int nin; bool has_bih, has_bhh; };
struct DensePlan {
    int G = 0;
    long long param_floats = 0;
    DenseLayerOff layer[TTRNN_MAX_LAYERS];
};
// parameter blob, per layer: [W_ih (G*H x I)] [b_ih (G*H): GRU with bias only] [W_hh (G*H x H)] [b_hh (G*H) with bias]
// (LSTMCell: input_weights has no bias, lstm.py:17-21; GRUCell: both carry `bias`, gru.py:19-23)
int build_dense_plan(const ttrnn_dense_desc *d, DensePlan *dp) {
    if (!d) return fail("null descriptor");
    if (d->cell != TTRNN_CELL_LSTM && d->cell != TTRNN_CELL_GRU) return fail("unknown cell kind %d", d->cell);
    if (d->num_layers < 1 || d->num_layers > TTRNN_MAX_LAYERS) return fail("num_layers %d out of range", d->num_layers);
    if (d->input_size < 1 || d->hidden_size < 1 || d->batch < 1 || d->seq_len < 1) return fail("sizes must be positive");
    if (d->hidden_size % 128 != 0)
        return fail("dense cells: hidden_size must be a multiple of 128 (the GEMM tiles are 128 columns wide), got %d", d->hidden_size);
    dp->G = gates_of(d->cell);
    const long long GH = (long long)dp->G * d->hidden_size;
    long long off = 0;
    for (int l = 0; l < d->num_layers; ++l) {
        DenseLayerOff &o = dp->layer[l];
        o.nin = l == 0 ? d->input_size : d->hidden_size;
        o.has_bih = d->has_bias && d->cell == TTRNN_CELL_GRU;
        o.has_bhh = d->has_bias != 0;
        o.w_ih = off; off += GH * o.nin;
        o.b_ih = off; if (o.has_bih) off += GH;
        o.w_hh = off; off += GH * d->hidden_size;
        o.b_hh = off; if (o.has_bhh) off += GH;
    }
    dp->param_floats = off;
    return 0;
}
struct DenseLayout {
    long long BTH, BTG, BH;
    long long sv_hs, sv_cs, sv_a, sv_u, sv_total;      // saved: inner-layer outputs, c states, a = W_ih x, u = W_hh h (per layer)
    long long s_w, s_dh, s_part, s_total;              // scratch: weight splits / transposes, dh carries, reduction partials
    long long wmax;
};
void build_dense_layout(const ttrnn_dense_desc *d, const DensePlan &dp, DenseLayout *lo) {
    const long long B = d->batch, T = d->seq_len, H = d->hidden_size, L = d->num_layers, GH = (long long)dp.G * H;
    const long long Imax = d->input_size > H ? d->input_size : H;
    lo->BTH = B * T * H; lo->BTG = B * T * GH; lo->BH = B * H;
    long long o = 0;
    lo->sv_hs = o; o += r4((L - 1) * lo->BTH);
    lo->sv_cs = o; o += (d->cell == TTRNN_CELL_LSTM) ? r4(L * lo->BTH) : 0;
    lo->sv_a = o; o += r4(L * lo->BTG);
    lo->sv_u = o; o += r4(L * lo->BTG);
    lo->sv_total = o;
    lo->wmax = r4(GH * Imax);
    o = 0;
    lo->s_w = o; o += 8 * lo->wmax;                    // W_ih hi/lo, W_hh hi/lo, W^T + hi/lo (one side at a time), dW^T
    lo->s_dh = o; o += 6 * r4(lo->BH);                 // dh_gemm, dh_direct x 2 (ping-pong), dc, h zero pad, spare
    lo->s_part = o; o += kDenseMaxSplit * (lo->wmax + r4(GH)) + 2 * r4(GH);
    lo->s_total = o;
}
// y = x W^T (+ bias): rows GEMM on the tensor cores when it fits, else FFMA (needs W^T as K x N)
int dense_linear(const DevInfo &dv, long long rows, int rpb, const float *x, long long x_bstride, int K, const float *w_hi,
                 const float *w_lo, const float *wt, int N, const float *bias, float *y, long long y_bstride, bool grad,
                 cudaStream_t st) {
    return dense_rows_gemm(grad ? TTRNN_K_GEMM_DX : TTRNN_K_GEMM_FWD, dv, rows, rpb, x, x_bstride, K, wt, w_hi, w_lo, N, bias, nullptr,
                           y, y_bstride, grad, st);
}
// out[n] = sum over rows of m[r, n] (rows x N contiguous): split partial sums, then a fixed-order sum of the splits
int dense_colsum(const DevInfo &dv, const float *m, long long rows, int N, float *part, float *out, cudaStream_t st) {
    int nsplit = (int)((rows + 511) / 512);
    if (nsplit > kDenseMaxSplit) nsplit = kDenseMaxSplit;
    if (nsplit < 1) nsplit = 1;
    dim3 grid((N + 127) / 128, nsplit);
    ttd::k_colsum_part<<<grid, 128, 0, st>>>(m, rows, N, nsplit, part);
    ttg::k_sum_splits<<<(unsigned)((N / 4 + 255) / 256), 256, 0, st>>>(part, nsplit, N, N, out, 0);
    g_launches += 2;
    (void)dv;
    CU_CHECK(cudaGetLastError());
    return 0;
}
int transpose_to(const float *src, float *dst, int rows, int cols, cudaStream_t st) {
    dim3 grid((cols + 31) / 32, (rows + 31) / 32);
    ttg::k_transpose<<<grid, 256, 0, st>>>(src, dst, rows, cols);
    ++g_launches;
    CU_CHECK(cudaGetLastError());
    return 0;
}
}  // namespace

int64_t ttrnn_dense_rnn_param_count(const ttrnn_dense_desc *desc) {
    DensePlan dp;
    if (build_dense_plan(desc, &dp)) return -1;
    return dp.param_floats;
}

int ttrnn_dense_rnn_workspace_bytes(const ttrnn_dense_desc *desc, int64_t *saved_bytes, int64_t *scratch_bytes) {
    DensePlan dp;
    if (build_dense_plan(desc, &dp)) return 1;
    if (!saved_bytes || !scratch_bytes) return fail("null output pointer");
    DenseLayout lo;
    build_dense_layout(desc, dp, &lo);
    *saved_bytes = lo.sv_total * 4;
    *scratch_bytes = lo.s_total * 4;
    return 0;
}

static int dense_forward(const ttrnn_dense_desc *d, const StateMap &sm, const float *x, const float *h0, const float *c0,
                         const float *params, float *out, float *hT, float *cT, void *saved, void *scratch, void *stream) {
    t_opt = snapshot_options();
    DensePlan dp;
    if (build_dense_plan(d, &dp)) return 1;
    if (!x || !params || !out || !saved || !scratch) return fail("x, params, out, saved and scratch must be non-null");
    DevInfo dv;
    if (get_dev(&dv)) return 1;
    DenseLayout lo;
    build_dense_layout(d, dp, &lo);
    cudaStream_t st = (cudaStream_t)stream;
    const long long B = d->batch;
    const int T = d->seq_len, H = d->hidden_size, L = d->num_layers, G = dp.G, GH = G * H;
    const bool lstm = d->cell == TTRNN_CELL_LSTM;
    float *sv = (float *)saved, *sc = (float *)scratch;
    float *w_ih_hi = sc + lo.s_w, *w_ih_lo = w_ih_hi + lo.wmax, *w_hh_hi = w_ih_lo + lo.wmax, *w_hh_lo = w_hh_hi + lo.wmax;
    float *wt_ih = w_hh_lo + lo.wmax, *wt_hh = wt_ih + lo.wmax;
    long long blocks = (B * (long long)H + 255) / 256;
    if (blocks > (long long)dv.sms * 8) blocks = (long long)dv.sms * 8;
    for (int l = 0; l < L; ++l) {
        const DenseLayerOff &o = dp.layer[l];
        const float *lin = l == 0 ? x : sv + lo.sv_hs + (long long)(l - 1) * lo.BTH;
        float *lout = l == L - 1 ? out : sv + lo.sv_hs + (long long)l * lo.BTH;
        float *cs = lstm ? sv + lo.sv_cs + (long long)l * lo.BTH : nullptr;
        float *ab = sv + lo.sv_a + (long long)l * lo.BTG, *ub = sv + lo.sv_u + (long long)l * lo.BTG;
        const float *W_ih = params + o.w_ih, *W_hh = params + o.w_hh;
        const long long nih = (long long)GH * o.nin, nhh = (long long)GH * H;
        // both operand forms: TF32 hi / lo split of W (tensor cores) and W^T as K x N (FFMA fallback)
        if (o.nin % 4 == 0 && (split_tf32(W_ih, w_ih_hi, w_ih_lo, r4(nih), st) || transpose_to(W_ih, wt_ih, GH, o.nin, st))) return 1;
        if (split_tf32(W_hh, w_hh_hi, w_hh_lo, r4(nhh), st) || transpose_to(W_hh, wt_hh, GH, H, st)) return 1;
        // a = X W_ih^T (+ b_ih) for every timestep at once
        if (o.nin % 4 != 0) {
            long long gb = (B * (long long)T * GH + 255) / 256;
            if (gb > (long long)dv.sms * 16) gb = (long long)dv.sms * 16;
            ttd::k_smallk_fwd<<<(unsigned)gb, 256, 0, st>>>(lin, W_ih, o.has_bih ? params + o.b_ih : nullptr, ab, B * (long long)T, o.nin, GH);
            ++g_launches;
        } else if (dense_linear(dv, B * (long long)T, T, lin, (long long)T * o.nin, o.nin, w_ih_hi, w_ih_lo, wt_ih, GH,
                         o.has_bih ? params + o.b_ih : nullptr, ab, (long long)T * GH, false, st))
            return 1;
        const float *h0l = sm.init(h0, l), *c0l = sm.init(c0, l);
        for (int t = 0; t < T; ++t) {
            const float *hp = t == 0 ? h0l : lout + (long long)(t - 1) * H;
            const long long ldhp = t == 0 ? H : (long long)T * H;
            // u_t = h_{t-1} W_hh^T + b_hh  (h_{-1} = 0: u_0 = b_hh)
            if (hp) {
                if (dense_linear(dv, B, 1, hp, ldhp, H, w_hh_hi, w_hh_lo, wt_hh, GH,
                                 o.has_bhh ? params + o.b_hh : nullptr, ub + (long long)t * GH, (long long)T * GH, false, st))
                    return 1;
            } else {
                ttd::k_bias_rows<<<(unsigned)blocks, 256, 0, st>>>(o.has_bhh ? params + o.b_hh : nullptr, ub + (long long)t * GH,
                                                                   (long long)T * GH, B, GH);
                ++g_launches;
            }
            ttd::DenseStepArgs a;
            memset(&a, 0, sizeof a);
            a.B = B; a.H = H;
            a.a = ab + (long long)t * GH; a.lda = (long long)T * GH;
            a.u = ub + (long long)t * GH; a.ldu = (long long)T * GH;
            a.h_prev = hp; a.ldhp = ldhp;
            a.c_prev = t == 0 ? c0l : cs + (long long)(t - 1) * H; a.ldcp = t == 0 ? H : (long long)T * H;
            a.h = lout + (long long)t * H; a.ldh = (long long)T * H;
            a.c = lstm ? cs + (long long)t * H : nullptr; a.ldc = (long long)T * H;
            {
                KernelTimer tm(TTRNN_K_RNN_FWD, st);
                if (lstm) ttd::k_dense_cell_fwd<true><<<(unsigned)blocks, 256, 0, st>>>(a);
                else ttd::k_dense_cell_fwd<false><<<(unsigned)blocks, 256, 0, st>>>(a);
            }
            ++g_launches;
        }
        CU_CHECK(cudaGetLastError());
        float *hTl = sm.fin(hT, l, L), *cTl = sm.fin(cT, l, L);
        if (hTl) CU_CHECK(cudaMemcpy2DAsync(hTl, (size_t)H * 4, lout + (long long)(T - 1) * H, (size_t)T * H * 4, (size_t)H * 4, B,
                                            cudaMemcpyDeviceToDevice, st));
        if (lstm && cTl) CU_CHECK(cudaMemcpy2DAsync(cTl, (size_t)H * 4, cs + (long long)(T - 1) * H, (size_t)T * H * 4, (size_t)H * 4,
                                                    B, cudaMemcpyDeviceToDevice, st));
    }
    return 0;
}

static int dense_backward(const ttrnn_dense_desc *d, const StateMap &sm, const float *x, const float *h0, const float *c0,
                          const float *params, const float *out, void *saved, const float *d_out, const float *d_hT,
                          const float *d_cT, float *d_params, float *d_x, float *d_h0, float *d_c0, void *scratch, void *stream) {
    t_opt = snapshot_options();
    DensePlan dp;
    if (build_dense_plan(d, &dp)) return 1;
    if (!x || !params || !out || !saved || !scratch || !d_params) return fail("x, params, out, saved, scratch, d_params must be non-null");
    DevInfo dv;
    if (get_dev(&dv)) return 1;
    DenseLayout lo;
    build_dense_layout(d, dp, &lo);
    cudaStream_t st = (cudaStream_t)stream;
    const long long B = d->batch;
    const int T = d->seq_len, H = d->hidden_size, L = d->num_layers, G = dp.G, GH = G * H;
    const bool lstm = d->cell == TTRNN_CELL_LSTM;
    float *sv = (float *)saved, *sc = (float *)scratch;
    float *wT_hi = sc + lo.s_w, *wT_lo = wT_hi + lo.wmax, *wT = wT_lo + lo.wmax, *wplain_t = wT + lo.wmax, *dwt = wplain_t + lo.wmax;
    float *dh_gemm = sc + lo.s_dh, *dhd[2] = {dh_gemm + r4(lo.BH), dh_gemm + 2 * r4(lo.BH)}, *dcc = dh_gemm + 3 * r4(lo.BH);
    float *part = sc + lo.s_part, *pbias = part + kDenseMaxSplit * lo.wmax, *dbias = pbias + kDenseMaxSplit * r4(GH);
    long long blocks = (B * (long long)H + 255) / 256;
    if (blocks > (long long)dv.sms * 8) blocks = (long long)dv.sms * 8;
    // dW^T (K x GH) = sum over rows of A^T Bm, then transposed into the parameter layout (GH x K); db = column sums of Bm
    DenseIh D;
    memset(&D, 0, sizeof D);
    D.part = part; D.pbias = pbias; D.dwt = dwt; D.dbias = dbias;
    for (int l = L - 1; l >= 0; --l) {
        const DenseLayerOff &o = dp.layer[l];
        const float *lin = l == 0 ? x : sv + lo.sv_hs + (long long)(l - 1) * lo.BTH;
        const float *lout = l == L - 1 ? out : sv + lo.sv_hs + (long long)l * lo.BTH;
        const float *cs = lstm ? sv + lo.sv_cs + (long long)l * lo.BTH : nullptr;
        float *ab = sv + lo.sv_a + (long long)l * lo.BTG, *ub = sv + lo.sv_u + (long long)l * lo.BTG;
        // gradient wrt this layer's outputs: the caller's d_out for the last layer; for an inner layer the dX of the layer
        // above, which that layer wrote over its own (by then dead) `u` buffer, packed (B, T, H) at the front
        const float *dhs = l == L - 1 ? d_out : sv + lo.sv_u + (long long)(l + 1) * lo.BTG;
        const float *W_ih = params + o.w_ih, *W_hh = params + o.w_hh;
        const long long nhh = (long long)GH * H;
        // dh_{t-1} += du_t W_hh : rows GEMM with Bt = W_hh^T (H x GH)
        if (transpose_to(W_hh, wT, GH, H, st)) return 1;                         // wT = W_hh^T (H x GH)
        if (split_tf32(wT, wT_hi, wT_lo, r4(nhh), st)) return 1;
        const float *h0l = sm.init(h0, l), *c0l = sm.init(c0, l);
        const float *dhTl = sm.fin(d_hT, l, L), *dcTl = sm.fin(d_cT, l, L);
        for (int t = T - 1; t >= 0; --t) {
            ttd::DenseStepArgs a;
            memset(&a, 0, sizeof a);
            a.B = B; a.H = H;
            a.a = ab + (long long)t * GH; a.lda = (long long)T * GH;
            a.u = ub + (long long)t * GH; a.ldu = (long long)T * GH;
            a.h_prev = t == 0 ? h0l : lout + (long long)(t - 1) * H; a.ldhp = t == 0 ? H : (long long)T * H;
            a.c_prev = t == 0 ? c0l : (lstm ? cs + (long long)(t - 1) * H : nullptr); a.ldcp = t == 0 ? H : (long long)T * H;
            a.dout = dhs ? dhs + (long long)t * H : nullptr; a.lddo = (long long)T * H;
            a.first = t == T - 1;
            a.dh_gemm = a.first ? nullptr : dh_gemm;
            a.dh_direct = (a.first || lstm) ? nullptr : dhd[(t + 1) & 1];
            a.dh_T = a.first ? dhTl : nullptr;
            a.dc_T = a.first ? dcTl : nullptr;
            a.da = ab + (long long)t * GH; a.ldda = (long long)T * GH;
            a.du = ub + (long long)t * GH; a.lddu = (long long)T * GH;
            a.dh_direct_out = dhd[t & 1];
            a.dc = dcc;
            {
                KernelTimer tm(TTRNN_K_RNN_BWD, st);
                if (lstm) ttd::k_dense_cell_bwd<true><<<(unsigned)blocks, 256, 0, st>>>(a);
                else ttd::k_dense_cell_bwd<false><<<(unsigned)blocks, 256, 0, st>>>(a);
            }
            ++g_launches;
            if (t > 0 || (d_h0 && h0l)) {
                // dh_gemm = du_t W_hh
                if (dense_linear(dv, B, 1, ub + (long long)t * GH, (long long)T * GH, GH, wT_hi, wT_lo, W_hh, H, nullptr,
                                 dh_gemm, H, true, st))
                    return 1;
            }
        }
        CU_CHECK(cudaGetLastError());
        // gradient wrt the initial state: this layer's own block, or the sum over layers when the state is shared
        if (d_h0 && h0l) {
            ttd::k_add2<<<(unsigned)blocks, 256, 0, st>>>(dh_gemm, lstm ? nullptr : dhd[0], sc + lo.s_dh + 4 * r4(lo.BH), lo.BH);
            ++g_launches;
            if (axpy1(sc + lo.s_dh + 4 * r4(lo.BH), sm.init(d_h0, l), lo.BH, !sm.stride && l != L - 1, st)) return 1;
        }
        if (lstm && d_c0 && c0l && axpy1(dcc, sm.init(d_c0, l), lo.BH, !sm.stride && l != L - 1, st)) return 1;
        // dW_hh^T (H x GH) = sum_t h_{t-1}^T du_t ; db_hh = column sums of du (all T steps)
        {
            bool acc = false;
            if (T > 1) {
                if (dense_dw(dv, B * (long long)(T - 1), T - 1, lout, (long long)T * H, H, ub + GH, (long long)T * GH, GH, D, false, false, st))
                    return 1;
                acc = true;
            }
            if (h0l) {
                if (dense_dw(dv, B, 1, h0l, H, H, ub, (long long)T * GH, GH, D, acc, false, st)) return 1;
                acc = true;
            }
            if (acc) {
                if (transpose_to(dwt, d_params + o.w_hh, H, GH, st)) return 1;
            } else {
                CU_CHECK(cudaMemsetAsync(d_params + o.w_hh, 0, (size_t)nhh * 4, st));
            }
            if (o.has_bhh && dense_colsum(dv, ub, B * (long long)T, GH, part, d_params + o.b_hh, st)) return 1;
        }
        // dW_ih^T (I x GH) = X^T da ; db_ih = column sums of da
        if (o.nin % 4 != 0) {
            const long long rows = B * (long long)T;
            int nsplit = (int)((rows + 511) / 512);
            if (nsplit > kDenseMaxSplit) nsplit = kDenseMaxSplit;
            if ((long long)nsplit * GH * o.nin > kDenseMaxSplit * lo.wmax) return fail("dense cells: input_size %d unsupported", o.nin);
            dim3 grid((GH + 127) / 128, nsplit, o.nin);
            ttd::k_smallk_dw_part<<<grid, 128, 0, st>>>(ab, lin, rows, GH, o.nin, nsplit, part);
            const long long wn = r4((long long)GH * o.nin);
            if (((long long)GH * o.nin) % 4 != 0) return fail("dense cells: G*H*input_size must be a multiple of 4");
            ttg::k_sum_splits<<<(unsigned)((wn / 4 + 255) / 256), 256, 0, st>>>(part, nsplit, (long long)GH * o.nin, (long long)GH * o.nin,
                                                                                 d_params + o.w_ih, 0);
            g_launches += 2;
        } else {
            if (dense_dw(dv, B * (long long)T, T, lin, (long long)T * o.nin, o.nin, ab, (long long)T * GH, GH, D, false, false, st)) return 1;
            if (transpose_to(dwt, d_params + o.w_ih, o.nin, GH, st)) return 1;
        }
        if (o.has_bih && dense_colsum(dv, ab, B * (long long)T, GH, part, d_params + o.b_ih, st)) return 1;
        // dX = da W_ih (B, T, I): for l > 0 it is the upstream gradient of the layer below, written over this layer's dead
        // `u` buffer (packed (B, T, H) at its front); for l == 0 into the caller's d_x (if requested)
        float *dxl = l == 0 ? d_x : ub;
        if (dxl) {
            if (o.nin % 128 != 0)
                return fail("dense cells: the gradient wrt the input needs input_size %% 128 == 0 (got %d)", o.nin);
            if (transpose_to(W_ih, wT, GH, o.nin, st)) return 1;                // wT = W_ih^T (I x GH)
            if (split_tf32(wT, wT_hi, wT_lo, r4((long long)GH * o.nin), st)) return 1;
            if (dense_linear(dv, B * (long long)T, T, ab, (long long)T * GH, GH, wT_hi, wT_lo, W_ih, o.nin, nullptr, dxl,
                             (long long)T * o.nin, true, st))
                return 1;
        }
    }
    return 0;
}

// ---- GE2E head (SURVEY.md 8f-4) ------------------------------------------------------------------------------------
int ttrnn_dense_rnn_forward(const ttrnn_dense_desc *d, const float *x, const float *h0, const float *c0, const float *params,
                            float *out, float *hT, float *cT, void *saved, void *scratch, void *stream) {
    return dense_forward(d, StateMap(), x, h0, c0, params, out, hT, cT, saved, scratch, stream);
}
int ttrnn_dense_rnn_backward(const ttrnn_dense_desc *d, const float *x, const float *h0, const float *c0, const float *params,
                             const float *out, void *saved, const float *d_out, const float *d_hT, const float *d_cT,
                             float *d_params, float *d_x, float *d_h0, float *d_c0, void *scratch, void *stream) {
    return dense_backward(d, StateMap(), x, h0, c0, params, out, saved, d_out, d_hT, d_cT, d_params, d_x, d_h0, d_c0, scratch,
                          stream);
}
static int dense_state_map(const ttrnn_dense_desc *d, int32_t flags, StateMap *sm) {
    if (!d) return fail("null descriptor");
    if (flags & ~TTRNN_WS_LAYER_STATES) return fail("dense cells: unknown flags 0x%x (only TTRNN_WS_LAYER_STATES applies)", flags);
    if (flags & TTRNN_WS_LAYER_STATES) sm->stride = d->batch * (long long)d->hidden_size;
    return 0;
}
int ttrnn_dense_rnn_forward_ex(const ttrnn_dense_desc *d, const float *x, const float *h0, const float *c0, const float *params,
                               float *out, float *hT, float *cT, void *saved, void *scratch, void *stream, int32_t flags) {
    StateMap sm;
    if (dense_state_map(d, flags, &sm)) return 1;
    return dense_forward(d, sm, x, h0, c0, params, out, hT, cT, saved, scratch, stream);
}
int ttrnn_dense_rnn_backward_ex(const ttrnn_dense_desc *d, const float *x, const float *h0, const float *c0, const float *params,
                                const float *out, void *saved, const float *d_out, const float *d_hT, const float *d_cT,
                                float *d_params, float *d_x, float *d_h0, float *d_c0, void *scratch, void *stream, int32_t flags) {
    StateMap sm;
    if (dense_state_map(d, flags, &sm)) return 1;
    return dense_backward(d, sm, x, h0, c0, params, out, saved, d_out, d_hT, d_cT, d_params, d_x, d_h0, d_c0, scratch, stream);
}

int ttrnn_embed_forward(int64_t rows, int32_t E, const float *x, float *y, float *inv_norm, void *stream) {
    if (rows < 1 || E < 1) return fail("ttrnn_embed_forward: rows and E must be >= 1");
    if (!x || !y || !inv_norm) return fail("ttrnn_embed_forward: null operand");
    DevInfo dv;
    if (get_dev(&dv)) return 1;
    ge2e::k_embed_fwd<<<(unsigned)((rows + 7) / 8), ge2e::NT, 0, (cudaStream_t)stream>>>(x, y, inv_norm, (int)rows, E);
    ++g_launches;
    CU_CHECK(cudaGetLastError());
    return 0;
}

int ttrnn_embed_backward(int64_t rows, int32_t E, const float *x, const float *y, const float *inv_norm, const float *dy,
                         float *dx, void *stream) {
    if (rows < 1 || E < 1) return fail("ttrnn_embed_backward: rows and E must be >= 1");
    if (!x || !y || !inv_norm || !dy || !dx) return fail("ttrnn_embed_backward: null operand");
    DevInfo dv;
    if (get_dev(&dv)) return 1;
    ge2e::k_embed_bwd<<<(unsigned)((rows + 7) / 8), ge2e::NT, 0, (cudaStream_t)stream>>>(x, y, inv_norm, dy, dx, (int)rows, E);
    ++g_launches;
    CU_CHECK(cudaGetLastError());
    return 0;
}

// workspace layout (floats): c_incl S*E | n_incl S | c_excl S*U*E | n_excl S*U | sim B*S | prob B*S | row B | dsim B*S | row_dw B | row_db B
struct Ge2eWs {
    float *c_incl, *n_incl, *c_excl, *n_excl, *sim, *prob, *row, *dsim, *row_dw, *row_db;
    long long total;
};
static Ge2eWs ge2e_carve(float *base, long long S, long long U, long long E) {
    Ge2eWs w;
    const long long B = S * U;
    long long o = 0;
    auto take = [&](long long n) { float *p = base ? base + o : nullptr; o += r4(n); return p; };
    w.c_incl = take(S * E); w.n_incl = take(S); w.c_excl = take(B * E); w.n_excl = take(B);
    w.sim = take(B * S); w.prob = take(B * S); w.row = take(B); w.dsim = take(B * S); w.row_dw = take(B); w.row_db = take(B);
    w.total = o;
    return w;
}
static int ge2e_args_ok(int S, int U, int E) {
    if (S < 2 || U < 2 || E < 1) return fail("GE2E loss needs >= 2 speakers, >= 2 utterances per speaker and E >= 1 (got %d, %d, %d)", S, U, E);
    if ((long long)(E + S + 8) * 4 > 200 * 1024) return fail("GE2E loss: embedding size %d / %d speakers exceed the shared-memory staging", E, S);
    return 0;
}

int64_t ttrnn_ge2e_workspace_bytes(int32_t S, int32_t U, int32_t E) {
    if (ge2e_args_ok(S, U, E)) return -1;
    return ge2e_carve(nullptr, S, U, E).total * 4;
}

int ttrnn_ge2e_loss_forward(int32_t S, int32_t U, int32_t E, const float *embeds, const float *wb, float *loss,
                            float *sim_out, void *workspace, void *stream) {
    if (ge2e_args_ok(S, U, E)) return 1;
    if (!embeds || !wb || !loss || !workspace) return fail("ttrnn_ge2e_loss_forward: null operand");
    DevInfo dv;
    if (get_dev(&dv)) return 1;
    cudaStream_t st = (cudaStream_t)stream;
    Ge2eWs w = ge2e_carve((float *)workspace, S, U, E);
    const int B = S * U;
    ge2e::k_centroids<<<S, ge2e::NT, (size_t)(E + 8) * 4, st>>>(embeds, w.c_incl, w.n_incl, w.c_excl, w.n_excl, U, E);
    ge2e::k_sim_loss<<<B, ge2e::NT, (size_t)(E + S + 8) * 4, st>>>(embeds, w.c_incl, w.c_excl, wb, w.sim, w.prob, w.row, sim_out, S, U, E);
    ge2e::k_mean<<<1, ge2e::NT, 0, st>>>(w.row, B, loss);
    g_launches += 3;
    CU_CHECK(cudaGetLastError());
    return 0;
}

int ttrnn_ge2e_loss_backward(int32_t S, int32_t U, int32_t E, const float *embeds, const float *wb, const float *dloss,
                             void *workspace, float *d_embeds, float *d_wb, void *stream) {
    if (ge2e_args_ok(S, U, E)) return 1;
    if (!embeds || !wb || !dloss || !workspace || !d_embeds || !d_wb) return fail("ttrnn_ge2e_loss_backward: null operand");
    DevInfo dv;
    if (get_dev(&dv)) return 1;
    cudaStream_t st = (cudaStream_t)stream;
    Ge2eWs w = ge2e_carve((float *)workspace, S, U, E);
    const int B = S * U;
    ge2e::k_bwd_rows<<<B, ge2e::NT, (size_t)S * 4, st>>>(w.c_incl, w.c_excl, wb, w.sim, w.prob, dloss, w.dsim, d_embeds, w.row_dw,
                                                         w.row_db, S, U, E);
    ge2e::k_bwd_centroids<<<S, ge2e::NT, (size_t)(E + 8) * 4, st>>>(embeds, w.c_incl, w.n_incl, w.c_excl, w.n_excl, w.dsim, d_embeds,
                                                                 S, U, E);
    ge2e::k_sum<<<1, ge2e::NT, 0, st>>>(w.row_dw, B, d_wb);
    ge2e::k_sum<<<1, ge2e::NT, 0, st>>>(w.row_db, B, d_wb + 1);
    g_launches += 4;
    CU_CHECK(cudaGetLastError());
    return 0;
}

int ttrnn_ffma_probe(int32_t iters, float *sink, double *flops_out, void *stream) {
    DevInfo dv;
    if (get_dev(&dv)) return 1;
    if (!sink) return fail("sink must be a device pointer");
    const int ctas = dv.sms * 8;
    k_ffma_probe<<<ctas, TT_NTHREADS, 0, (cudaStream_t)stream>>>(iters, sink);
    CU_CHECK(cudaGetLastError());
    if (flops_out) *flops_out = 2.0 * 16 * 8 * (double)iters * TT_NTHREADS * ctas;
    return 0;
}

}  // extern "C"
