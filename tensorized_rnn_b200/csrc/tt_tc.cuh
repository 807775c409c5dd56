// Tensor-core path of the dense-route contractions (sm_100a only): tcgen05.mma kind::tf32 with an
// error-compensated 3xTF32 split, accumulators in TMEM, operands staged by TMA behind mbarrier rings.
//
// The two dense contractions of the ih projection / core-gradient accumulation (tt_gemm.cuh holds
// the FP32 FFMA versions) are plain large GEMMs:
//
//   k_tc_rows : C[r, n]  = sum_k A[r, k] Bt[n, k] (+ bias[n] + bias2[n])      forward xg, and dX = delta * W
//   k_tc_red  : P_s[m,n] = sum_{r in split s} A[r, m] B[r, n]                  dW^T = X^T delta (+ column sums = db)
//
// FP32 parity (1e-5 forward / 1e-4 gradients) excludes a single TF32 pass (2^-11 per product), so every
// FP32 operand x is split as x = hi + lo, hi = tf32_rna(x), lo = tf32_rna(x - hi), and the product is
// accumulated as hi*hi' + lo*hi' + hi*lo' (three MMAs per k-slice, FP32 accumulate in TMEM); the dropped
// lo*lo' term and the rounding of lo are O(2^-22) relative.
//
// Measured on B200 (tools/tc_gemm_test, round 2): the tensor core's FP32 accumulate TRUNCATES, so the error of
// one TMEM accumulator grows linearly with the number of MMAs chained into it (2e-7 at K = 40, 1.7e-6 at K = 256
// with all three products in one accumulator).  Therefore (i) the two small products go to their own accumulator
// (their truncation error is 2^-11 smaller) and only hi*hi' chains into the main one (K / 8 adds), and (ii) the
// reduction kernel, whose chains are thousands of k-slices long, promotes the main accumulator into FP32 registers
// (round-to-nearest adds on the CUDA cores) every RED_SEG k-blocks = 32 chained MMAs, double-buffered in TMEM so
// the tensor core keeps running during the promotion.
//
// Warp roles (one CTA per SM): one TMA producer thread, one MMA issuer thread, "splitter" warps that turn
// the raw FP32 tiles TMA delivered into the hi / lo operand tiles (k_tc_red: transposing them into the
// K-major 128-byte-swizzled layout on the way, because both of its operands are MN-major in memory),
// epilogue warps that read the accumulator with tcgen05.ld.  Small weight operands (Bt of k_tc_rows) are
// split once per call in global memory and arrive by TMA as ready hi / lo tiles.
//
// Operand tiles are the canonical K-major SWIZZLE_128B layout: 32 FP32 (128 B) per row, 8-row groups of
// 1024 B, 16-byte chunk index XOR (row & 7).  One MMA consumes 8 k-values (32 B): the descriptor start
// address advances by 32 B per k-slice.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "tt_umma.cuh"

namespace ttc {

// -DTC_PROBE (tools/tc_gemm_test only): clock64 around every wait of the MMA issuer of one CTA
#ifdef TC_PROBE
inline long long *&tc_probe_buf() { static long long *p = nullptr; return p; }
#define PROBE(acc_, stmt) tq = clock64(); stmt; acc_ += clock64() - tq;
#else
#define PROBE(acc_, stmt) stmt;
#endif

constexpr int BM = 128, BN = 128, BK = 32;
constexpr int TILE_BYTES = BM * BK * 4;          // 16 KiB: one 128 x 32 FP32 operand tile
constexpr int NT = 320;                          // 10 warps

// ---- ragged row geometry (time-chunk views of (B, T, width) tensors) ------------------------------
// flattened row r = b * rpb + t lives at p + b * bstride + t * ld.  A tile / k-block of the row dimension is a TMA
// box of rb rows along t and nbx batch entries along b:
//   rpb >= cap : rb = cap, nbx = 1, tpb = ceil(rpb / cap) boxes per batch entry (the last one partly out of bounds)
//   rpb <  cap : rb = rpb, nbx = cap / rpb, tpb = 1
struct RagBox {
    int rpb, nb, rb, nbx, tpb;
    long long nboxes;            // ceil(nb / nbx) * tpb
};
inline RagBox make_ragbox(long long rpb, long long nb, int cap) {
    RagBox g;
    g.rpb = (int)rpb; g.nb = (int)nb;
    if (rpb >= cap) { g.rb = cap; g.nbx = 1; g.tpb = (int)((rpb + cap - 1) / cap); }
    else { g.rb = (int)rpb; g.nbx = (int)(cap / rpb); g.tpb = 1; }
    g.nboxes = ((nb + g.nbx - 1) / g.nbx) * g.tpb;
    return g;
}

// one k-block (BK = 32 k-values, `nks` slices of 8) of the compensated product: hi*hi' into the main accumulator,
// lo*hi' + hi*lo' into the small-term accumulator.
// Measured on B200 (tools/mma_rate_probe, round 2): back-to-back kind::tf32 MMAs into ONE 128 x 128 accumulator dispatch
// every 67.5 clk (A from TMEM) / 77 clk (A from shared memory), but every change of accumulator between two consecutive
// MMAs costs ~55 clk more (the per-k-slice order small, small, main ran at 104 / 117 clk per MMA).  So the MMAs of a k-block
// are grouped by accumulator, and `main_first` alternates between k-blocks: one accumulator change per k-block.
__device__ __forceinline__ void issue_block_3x(uint32_t d_main, uint32_t d_small, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi,
                                               uint32_t b_lo, int nks, uint32_t idesc, bool first_main, bool first_small,
                                               bool main_first) {
    const uint64_t dah = umma_desc_sw128(a_hi), dal = umma_desc_sw128(a_lo);
    const uint64_t dbh = umma_desc_sw128(b_hi), dbl = umma_desc_sw128(b_lo);
    for (int pass = 0; pass < 2; ++pass) {
        if ((pass == 0) == main_first) {
            for (int ks = 0; ks < nks; ++ks) {
                const uint64_t o = (uint64_t)(ks * 2);              // 32 B per k-slice, in 16-byte units
                umma_tf32(d_main, dah + o, dbh + o, idesc, (first_main && ks == 0) ? 0u : 1u);
            }
        } else {
            for (int ks = 0; ks < nks; ++ks) {
                const uint64_t o = (uint64_t)(ks * 2);
                umma_tf32(d_small, dal + o, dbh + o, idesc, (first_small && ks == 0) ? 0u : 1u);
                umma_tf32(d_small, dah + o, dbl + o, idesc, 1u);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// hi / lo split of a small weight matrix in global memory (once per call)
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_split_tf32(const float *__restrict__ src, float *__restrict__ hi,
                                                     float *__restrict__ lo, long long n4) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
        const float4 v = __ldg(reinterpret_cast<const float4 *>(src) + i);
        float4 h, l;
        split4(v, h, l);
        reinterpret_cast<float4 *>(hi)[i] = h;
        reinterpret_cast<float4 *>(lo)[i] = l;
    }
}

// ---------------------------------------------------------------------------------------------------
// k_tc_rows:  C[r, n] = sum_k A[r, k] Bt[n, k] (+ bias[n] + bias2[n])
//   A  : ragged rows x K (FP32; TMA box {32 k, rb, nbx}, SWIZZLE_128B -> the K-major operand layout directly)
//   Bt : N x K, pre-split into hi / lo copies in global memory
//   persistent CTAs over (row tile, 128-column tile); TMEM holds two (main, small-term) pairs of 128 x 128 accumulators
//   so that the epilogue of one tile overlaps the main loop of the next
// warps 0-7: splitters (A tile -> hi in place + lo), 8-11: epilogue, 12: TMA producer, 13: MMA issuer + TMEM allocator
// (eight splitter warps: with four, one warp per scheduler walked the whole split chain of a k-block and the tensor pipe
// waited for it)
// ---------------------------------------------------------------------------------------------------
constexpr int ROWS_STAGES = 3;
constexpr int ROWS_NT = 448;                     // 14 warps
constexpr int ROWS_STAGE_BYTES = 4 * TILE_BYTES;             // A hi (raw lands here), A lo, Bt hi, Bt lo
constexpr int ROWS_SMEM = ROWS_STAGES * ROWS_STAGE_BYTES + 1024 /*alignment slack*/ + 256 /*barriers*/;
static_assert(ROWS_SMEM >= TMEM_EXCLUSIVE_SMEM, "TMEM co-residence rule");

struct TcRowsArgs {
    RagBox g;                // row tiles (cap 128)
    int K, N, tiles_n;
    long long ntiles;        // g.nboxes * tiles_n
    float *c;                // ragged rows x N, same (rpb, nb) geometry as A
    long long c_bstride;
    int c_ld;
    const float *bias, *bias2;
#ifdef TC_PROBE
    long long *probe;
#endif
};

__global__ void __launch_bounds__(ROWS_NT, 1)
k_tc_rows(const __grid_constant__ TcRowsArgs g, const __grid_constant__ CUtensorMap tmA,
          const __grid_constant__ CUtensorMap tmBhi, const __grid_constant__ CUtensorMap tmBlo) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bars = base + ROWS_STAGES * ROWS_STAGE_BYTES;
    // barriers (8 B each): full[s], split[s], empty[s], tmem_full[2], tmem_empty[2]; then the TMEM base slot
    auto bar_full = [&](int s) { return bars + 8u * s; };
    auto bar_split = [&](int s) { return bars + 8u * (ROWS_STAGES + s); };
    auto bar_empty = [&](int s) { return bars + 8u * (2 * ROWS_STAGES + s); };
    auto bar_tfull = [&](int a) { return bars + 8u * (3 * ROWS_STAGES + a); };
    auto bar_tempty = [&](int a) { return bars + 8u * (3 * ROWS_STAGES + 2 + a); };
    const uint32_t tmem_slot = bars + 8u * (3 * ROWS_STAGES + 4);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int s = 0; s < ROWS_STAGES; ++s) {
            mbar_init(bar_full(s), 1);
            mbar_init(bar_split(s), 256);
            mbar_init(bar_empty(s), 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(bar_tfull(a), 1);
            mbar_init(bar_tempty(a), 128);
        }
        fence_barrier_init();
    }
    if (warp == 13) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

    const int nkb = (g.K + BK - 1) / BK;
    const uint32_t idesc = umma_idesc_tf32(BM, BN);

    if (warp == 12) {
        // ---------------- TMA producer ----------------
        if (elect_one()) {
            tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmBhi); tma_prefetch_desc(&tmBlo);
            long long it = 0;
            for (long long tile = blockIdx.x; tile < g.ntiles; tile += gridDim.x) {
                const long long box = tile / g.tiles_n;
                const int n0 = (int)(tile % g.tiles_n) * BN;
                const int b0 = (int)(box / g.g.tpb) * g.g.nbx, t0 = (int)(box % g.g.tpb) * g.g.rb;
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int s = (int)(it % ROWS_STAGES);
                    const uint32_t ph = (uint32_t)((it / ROWS_STAGES) & 1);
                    mbar_wait(bar_empty(s), ph ^ 1u);
                    const uint32_t st = base + s * ROWS_STAGE_BYTES;
                    mbar_arrive_expect_tx(bar_full(s), (uint32_t)(g.g.rb * g.g.nbx * BK * 4 + 2 * TILE_BYTES));
                    tma_load_3d(st, &tmA, bar_full(s), kb * BK, t0, b0);
                    tma_load_3d(st + 2 * TILE_BYTES, &tmBhi, bar_full(s), kb * BK, n0, 0);
                    tma_load_3d(st + 3 * TILE_BYTES, &tmBlo, bar_full(s), kb * BK, n0, 0);
                }
            }
        }
    } else if (warp == 13) {
        // ---------------- MMA issuer ----------------
        if (elect_one()) {
            long long it = 0, nt = 0;
            for (long long tile = blockIdx.x; tile < g.ntiles; tile += gridDim.x, ++nt) {
                const int acc = (int)(nt & 1);
                mbar_wait(bar_tempty(acc), (uint32_t)(((nt >> 1) & 1) ^ 1));
                tc_fence_after();
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int s = (int)(it % ROWS_STAGES);
                    const uint32_t ph = (uint32_t)((it / ROWS_STAGES) & 1);
                    mbar_wait(bar_full(s), ph);
                    mbar_wait(bar_split(s), ph);
                    tc_fence_after();
                    const uint32_t st = base + s * ROWS_STAGE_BYTES;
                    const int krem = g.K - kb * BK;
                    const int nks = krem >= BK ? BK / 8 : (krem + 7) / 8;
                    issue_block_3x(tmem_base + acc * 2 * BN, tmem_base + acc * 2 * BN + BN, st, st + TILE_BYTES,
                                   st + 2 * TILE_BYTES, st + 3 * TILE_BYTES, nks, idesc, kb == 0, kb == 0, (kb & 1) != 0);
                    umma_commit(bar_empty(s));
                }
                umma_commit(bar_tfull(acc));
            }
        }
    } else if (warp < 8) {
        // ---------------- splitters: A tile -> hi (in place) + lo ----------------
        long long it = 0;
        for (long long tile = blockIdx.x; tile < g.ntiles; tile += gridDim.x) {
            for (int kb = 0; kb < nkb; ++kb, ++it) {
                const int s = (int)(it % ROWS_STAGES);
                const uint32_t ph = (uint32_t)((it / ROWS_STAGES) & 1);
                mbar_wait(bar_full(s), ph);
                uint8_t *st = smem_raw + (base - smem_u32(smem_raw)) + s * ROWS_STAGE_BYTES;
                float4 *ah = reinterpret_cast<float4 *>(st), *al = reinterpret_cast<float4 *>(st + TILE_BYTES);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int idx = threadIdx.x + 256 * j;
                    float4 h, l;
                    split4(ah[idx], h, l);
                    ah[idx] = h;
                    al[idx] = l;
                }
                fence_proxy_async();
                mbar_arrive(bar_split(s));
            }
        }
    } else {
        // ---------------- epilogue: TMEM -> registers -> (+ bias) -> global ----------------
        const int q = warp - 8;                        // TMEM lane quarter of this warp (warp % 4)
        const int i = q * 32 + lane;                   // row of the tile
        const int bi = i / g.g.rb, ti = i - bi * g.g.rb;
        long long nt = 0;
        for (long long tile = blockIdx.x; tile < g.ntiles; tile += gridDim.x, ++nt) {
            const int acc = (int)(nt & 1);
            const long long box = tile / g.tiles_n;
            const int n0 = (int)(tile % g.tiles_n) * BN;
            const int b = (int)(box / g.g.tpb) * g.g.nbx + bi, t = (int)(box % g.g.tpb) * g.g.rb + ti;
            const bool ok = bi < g.g.nbx && b < g.g.nb && t < g.g.rpb;
            float *crow = g.c + (long long)b * g.c_bstride + (long long)t * g.c_ld + n0;
            mbar_wait(bar_tfull(acc), (uint32_t)((nt >> 1) & 1));
            tc_fence_after();
#pragma unroll 1
            for (int cc = 0; cc < BN / 32; ++cc) {
                float v[32], w[32];
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * 2 * BN + cc * 32), v);
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * 2 * BN + BN + cc * 32), w);
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] += w[j];
                if (ok) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        float4 o = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                        if (g.bias) {
                            const float4 bb = __ldg(reinterpret_cast<const float4 *>(g.bias + n0 + cc * 32) + j);
                            o.x += bb.x; o.y += bb.y; o.z += bb.z; o.w += bb.w;
                        }
                        if (g.bias2) {
                            const float4 bb = __ldg(reinterpret_cast<const float4 *>(g.bias2 + n0 + cc * 32) + j);
                            o.x += bb.x; o.y += bb.y; o.z += bb.z; o.w += bb.w;
                        }
                        reinterpret_cast<float4 *>(crow + cc * 32)[j] = o;
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(bar_tempty(acc));
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 13) tmem_dealloc(tmem_base, 512);
}

// ---------------------------------------------------------------------------------------------------
// k_tc_rows_ts: k_tc_rows with the A operand in TMEM (tcgen05.mma "TS" form), the default.  k_tc_rows moves 192 KB through
// the shared-memory port per k-block (TMA 48, split load 16 + stores 32, three MMAs per k-slice reading A and B: 96), which
// is what bounds it; here row m of the raw A tile is split into TMEM lane m (tcgen05.st) and only Bt is read from shared
// memory by the MMAs: 112 KB per k-block, and a fourth TMA stage fits.
// TMEM columns: [0,128) [128,256) main accumulators (double-buffered across tiles), [256,384) small terms (single: the
// epilogue reads it first and hands it back before it touches the main accumulator), [384,512) two A stages (hi 32 | lo 32).
// warps 0-3: A splitters; 8-15: epilogue (lane quarter = warp % 4, 64 columns each); 16: TMA; 17: MMA issuer + TMEM allocator
// GRAD: the lo term is left unrounded (gradient tolerance 1e-4; see split4_trunc)
// ---------------------------------------------------------------------------------------------------
constexpr int RWT_STAGES = 4;
constexpr int RWT_NT = 576;
constexpr int RWT_STAGE_BYTES = 3 * TILE_BYTES;              // raw A, Bt hi, Bt lo
constexpr int RWT_SMEM = RWT_STAGES * RWT_STAGE_BYTES + 1024 + 256;
static_assert(RWT_SMEM >= TMEM_EXCLUSIVE_SMEM, "TMEM co-residence rule");

template <bool GRAD>
__global__ void __launch_bounds__(RWT_NT, 1)
k_tc_rows_ts(const __grid_constant__ TcRowsArgs g, const __grid_constant__ CUtensorMap tmA,
             const __grid_constant__ CUtensorMap tmBhi, const __grid_constant__ CUtensorMap tmBlo) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t *gbase = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t bars = base + RWT_STAGES * RWT_STAGE_BYTES;
    // full[s] (TMA landed), empty[s] (MMAs of the stage done + raw A consumed), aready[o] / afree[o] (A operand stage in
    // TMEM), tfull[a] / tempty[a] (main accumulator), sfree (small-term accumulator read by the epilogue)
    auto bar_full = [&](int s) { return bars + 8u * s; };
    auto bar_empty = [&](int s) { return bars + 8u * (RWT_STAGES + s); };
    auto bar_aready = [&](int o) { return bars + 8u * (2 * RWT_STAGES + o); };
    auto bar_afree = [&](int o) { return bars + 8u * (2 * RWT_STAGES + 2 + o); };
    auto bar_tfull = [&](int a) { return bars + 8u * (2 * RWT_STAGES + 4 + a); };
    auto bar_tempty = [&](int a) { return bars + 8u * (2 * RWT_STAGES + 6 + a); };
    const uint32_t bar_sfree = bars + 8u * (2 * RWT_STAGES + 8);
    const uint32_t tmem_slot = bars + 8u * (2 * RWT_STAGES + 9);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int s = 0; s < RWT_STAGES; ++s) { mbar_init(bar_full(s), 1); mbar_init(bar_empty(s), 129); }
        for (int o = 0; o < 2; ++o) { mbar_init(bar_aready(o), 128); mbar_init(bar_afree(o), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(bar_tfull(a), 1); mbar_init(bar_tempty(a), 256); }
        mbar_init(bar_sfree, 256);
        fence_barrier_init();
    }
    if (warp == 17) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
    constexpr uint32_t A_COL0 = 3 * BN;
    const int nkb = (g.K + BK - 1) / BK;

    if (warp == 16) {
        // ---------------- TMA producer ----------------
        if (elect_one()) {
            tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmBhi); tma_prefetch_desc(&tmBlo);
            long long it = 0;
            for (long long tile = blockIdx.x; tile < g.ntiles; tile += gridDim.x) {
                const long long box = tile / g.tiles_n;
                const int n0 = (int)(tile % g.tiles_n) * BN;
                const int b0 = (int)(box / g.g.tpb) * g.g.nbx, t0 = (int)(box % g.g.tpb) * g.g.rb;
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int s = (int)(it % RWT_STAGES);
                    const uint32_t ph = (uint32_t)((it / RWT_STAGES) & 1);
                    mbar_wait(bar_empty(s), ph ^ 1u);
                    const uint32_t st = base + s * RWT_STAGE_BYTES;
                    mbar_arrive_expect_tx(bar_full(s), (uint32_t)(g.g.rb * g.g.nbx * BK * 4 + 2 * TILE_BYTES));
                    tma_load_3d(st, &tmA, bar_full(s), kb * BK, t0, b0);
                    tma_load_3d(st + TILE_BYTES, &tmBhi, bar_full(s), kb * BK, n0, 0);
                    tma_load_3d(st + 2 * TILE_BYTES, &tmBlo, bar_full(s), kb * BK, n0, 0);
                }
            }
        }
    } else if (warp == 17) {
        // ---------------- MMA issuer ----------------
        if (elect_one()) {
            const uint32_t idesc = umma_idesc_tf32(BM, BN);
            const uint32_t d_small = tmem_base + 2 * BN;
            long long it = 0, nt = 0;
#ifdef TC_PROBE
            long long w_tempty = 0, w_full = 0, w_aready = 0, w_sfree = 0, t_issue = 0, tq;
            const long long t_begin = clock64();
#endif
            for (long long tile = blockIdx.x; tile < g.ntiles; tile += gridDim.x, ++nt) {
                const int acc = (int)(nt & 1);
                const uint32_t d_main = tmem_base + acc * BN;
                PROBE(w_tempty, mbar_wait(bar_tempty(acc), (uint32_t)(((nt >> 1) & 1) ^ 1)))
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int s = (int)(it % RWT_STAGES), o = (int)(it & 1);
                    PROBE(w_full, mbar_wait(bar_full(s), (uint32_t)((it / RWT_STAGES) & 1)))
                    PROBE(w_aready, mbar_wait(bar_aready(o), (uint32_t)((it >> 1) & 1)))
                    tc_fence_after();
#ifdef TC_PROBE
                    const long long ti0 = clock64();
#endif
                    const uint32_t st = base + s * RWT_STAGE_BYTES;
                    const uint64_t dbh = umma_desc_sw128(st + TILE_BYTES), dbl = umma_desc_sw128(st + 2 * TILE_BYTES);
                    const uint32_t a_hi = tmem_base + A_COL0 + (uint32_t)o * 64u, a_lo = a_hi + 32u;
                    const int krem = g.K - kb * BK;
                    const int nks = krem >= BK ? BK / 8 : (krem + 7) / 8;
                    // grouped by accumulator (see issue_block_3x); the first k-block of a tile starts with the main products so
                    // that the tensor core has work while the epilogue of the previous tile still reads the small-term accumulator
                    const bool main_first = (kb & 1) == 0;
                    for (int pass = 0; pass < 2; ++pass) {
                        if ((pass == 0) == main_first) {
                            for (int ks = 0; ks < nks; ++ks)
                                umma_tf32_ts(d_main, a_hi + ks * 8, dbh + (uint64_t)(ks * 2), idesc, (kb == 0 && ks == 0) ? 0u : 1u);
                        } else {
                            if (kb == 0) {
                                PROBE(w_sfree, mbar_wait(bar_sfree, (uint32_t)((nt & 1) ^ 1)))
                                tc_fence_after();
                            }
                            for (int ks = 0; ks < nks; ++ks) {
                                umma_tf32_ts(d_small, a_lo + ks * 8, dbh + (uint64_t)(ks * 2), idesc, (kb == 0 && ks == 0) ? 0u : 1u);
                                umma_tf32_ts(d_small, a_hi + ks * 8, dbl + (uint64_t)(ks * 2), idesc, 1u);
                            }
                        }
                    }
                    umma_commit(bar_empty(s));
                    umma_commit(bar_afree(o));
#ifdef TC_PROBE
                    t_issue += clock64() - ti0;
#endif
                }
                umma_commit(bar_tfull(acc));
            }
#ifdef TC_PROBE
            if (blockIdx.x == 3 && g.probe) {
                g.probe[0] = clock64() - t_begin; g.probe[1] = w_tempty; g.probe[2] = w_full; g.probe[3] = w_aready;
                g.probe[4] = w_sfree; g.probe[5] = t_issue; g.probe[6] = it;
            }
#endif
        }
    } else if (warp < 4) {
        // ---------------- A splitters: row m of the raw K-major (128-byte swizzled) tile -> TMEM lane m ----------------
        const int m = warp * 32 + lane;
        long long it = 0;
        for (long long tile = blockIdx.x; tile < g.ntiles; tile += gridDim.x) {
            for (int kb = 0; kb < nkb; ++kb, ++it) {
                const int s = (int)(it % RWT_STAGES), o = (int)(it & 1);
                mbar_wait(bar_full(s), (uint32_t)((it / RWT_STAGES) & 1));
                const uint8_t *row = gbase + s * RWT_STAGE_BYTES + m * 128;
                float hi[32], lo[32];
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const float4 v = *reinterpret_cast<const float4 *>(row + ((c ^ (m & 7)) << 4));
                    float4 h, l;
                    if (GRAD) split4_trunc(v, h, l); else split4(v, h, l);
                    hi[4 * c] = h.x; hi[4 * c + 1] = h.y; hi[4 * c + 2] = h.z; hi[4 * c + 3] = h.w;
                    lo[4 * c] = l.x; lo[4 * c + 1] = l.y; lo[4 * c + 2] = l.z; lo[4 * c + 3] = l.w;
                }
                mbar_wait(bar_afree(o), (uint32_t)(((it >> 1) & 1) ^ 1));
                tc_fence_after();
                const uint32_t ta = tmem_base + ((uint32_t)(warp * 32) << 16) + A_COL0 + (uint32_t)o * 64u;
                tmem_st32(ta, hi);
                tmem_st32(ta + 32, lo);
                tmem_wait_st();
                mbar_arrive(bar_empty(s));                   // raw A consumed (after the stores that take the loaded registers)
                tc_fence_before();
                mbar_arrive(bar_aready(o));
            }
        }
    } else if (warp >= 8 && warp < 16) {
        // ---------------- epilogue: small terms first (hand the accumulator back), then main + small (+ bias) -> global ------
        const int q = warp & 3, ch = (warp - 8) >> 2;
        const int i = q * 32 + lane;
        const int bi = i / g.g.rb, ti = i - bi * g.g.rb;
        const uint32_t tl = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ch * 64);
        long long nt = 0;
        for (long long tile = blockIdx.x; tile < g.ntiles; tile += gridDim.x, ++nt) {
            const int acc = (int)(nt & 1);
            const long long box = tile / g.tiles_n;
            const int n0 = (int)(tile % g.tiles_n) * BN + ch * 64;
            const int b = (int)(box / g.g.tpb) * g.g.nbx + bi, t = (int)(box % g.g.tpb) * g.g.rb + ti;
            const bool ok = bi < g.g.nbx && b < g.g.nb && t < g.g.rpb;
            float *crow = g.c + (long long)b * g.c_bstride + (long long)t * g.c_ld + n0;
            mbar_wait(bar_tfull(acc), (uint32_t)((nt >> 1) & 1));
            tc_fence_after();
            float w[64];
            {
                float v[32];
                tmem_ld32(tl + (uint32_t)(2 * BN), v);
#pragma unroll
                for (int j = 0; j < 32; ++j) w[j] = v[j];
                tmem_ld32(tl + (uint32_t)(2 * BN + 32), v);
#pragma unroll
                for (int j = 0; j < 32; ++j) w[32 + j] = v[j];
            }
            tc_fence_before();
            mbar_arrive(bar_sfree);
#pragma unroll
            for (int cc = 0; cc < 2; ++cc) {
                float v[32];
                tmem_ld32(tl + (uint32_t)(acc * BN + cc * 32), v);
                if (cc == 1) {                               // both halves of the main accumulator are in registers
                    tc_fence_before();
                    mbar_arrive(bar_tempty(acc));
                }
                if (ok) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        float4 o4 = make_float4(v[4 * j] + w[cc * 32 + 4 * j], v[4 * j + 1] + w[cc * 32 + 4 * j + 1],
                                                v[4 * j + 2] + w[cc * 32 + 4 * j + 2], v[4 * j + 3] + w[cc * 32 + 4 * j + 3]);
                        if (g.bias) {
                            const float4 bb = __ldg(reinterpret_cast<const float4 *>(g.bias + n0 + cc * 32) + j);
                            o4.x += bb.x; o4.y += bb.y; o4.z += bb.z; o4.w += bb.w;
                        }
                        if (g.bias2) {
                            const float4 bb = __ldg(reinterpret_cast<const float4 *>(g.bias2 + n0 + cc * 32) + j);
                            o4.x += bb.x; o4.y += bb.y; o4.z += bb.z; o4.w += bb.w;
                        }
                        reinterpret_cast<float4 *>(crow + cc * 32)[j] = o4;
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 17) tmem_dealloc(tmem_base, 512);
}

// ---------------------------------------------------------------------------------------------------
// k_tc_red:  part[s][m, n] = sum_{r in k-blocks of split s} A[r, m] B[r, n];  pbias[s][n] = sum_r B[r, n]
//   A : ragged rows x M, B : ragged rows x N (FP32).  The contraction runs over ROWS, so both operands are MN-major
//   in memory: TMA delivers raw [32 rows][128] tiles (no swizzle) and the splitter warps write the hi / lo operand tiles
//   transposed into the K-major SWIZZLE_128B layout.  One 128 x 128 output tile per CTA.
//   TMEM: main accumulator x 2 (segments of RED_SEG k-blocks, promoted into FP32 registers by the drain warps while the
//   tensor core fills the other buffer) + one small-term accumulator that lives for the whole CTA.
// warps 0-7: splitters; 8-15: drain (promotion + final store); 16: TMA producer; 17: MMA issuer + TMEM allocator
// ---------------------------------------------------------------------------------------------------
constexpr int RED_NT = 576;
constexpr int RED_SEG = 8;                                   // k-blocks per TMEM segment: 32 chained hi*hi' MMAs (~6e-7)
constexpr int RED_RAW_STAGES = 3, RED_OP_STAGES = 2;
constexpr int RED_RAW_BYTES = 2 * TILE_BYTES;                // raw A [32][128], raw B [32][128]
constexpr int RED_OP_BYTES = 4 * TILE_BYTES;                 // A hi, A lo, B hi, B lo
constexpr int RED_SMEM = RED_RAW_STAGES * RED_RAW_BYTES + RED_OP_STAGES * RED_OP_BYTES + 1024 + 256 + 2 * 128 * 4;
static_assert(RED_SMEM >= TMEM_EXCLUSIVE_SMEM, "TMEM co-residence rule");

struct TcRedArgs {
    RagBox g;                // k-blocks of the row dimension (cap 32)
    int M, N, tiles_m, tiles_n;
    long long per;           // k-blocks per split
    int nsplit;
    float *part;             // [nsplit][M][N]
    float *pbias;            // [nsplit][N] or null
#ifdef TC_PROBE
    long long *probe;
#endif
};

__global__ void __launch_bounds__(RED_NT, 1)
k_tc_red(const __grid_constant__ TcRedArgs g, const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t *gbase = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t raw0 = base, op0 = base + RED_RAW_STAGES * RED_RAW_BYTES;
    const uint32_t bars = op0 + RED_OP_STAGES * RED_OP_BYTES;
    auto bar_rfull = [&](int s) { return bars + 8u * s; };
    auto bar_rempty = [&](int s) { return bars + 8u * (RED_RAW_STAGES + s); };
    auto bar_ofull = [&](int s) { return bars + 8u * (2 * RED_RAW_STAGES + s); };
    auto bar_oempty = [&](int s) { return bars + 8u * (2 * RED_RAW_STAGES + RED_OP_STAGES + s); };
    auto bar_afull = [&](int a) { return bars + 8u * (2 * RED_RAW_STAGES + 2 * RED_OP_STAGES + a); };
    auto bar_aempty = [&](int a) { return bars + 8u * (2 * RED_RAW_STAGES + 2 * RED_OP_STAGES + 2 + a); };
    const uint32_t tmem_slot = bars + 8u * (2 * RED_RAW_STAGES + 2 * RED_OP_STAGES + 4);
    float *bias_red = reinterpret_cast<float *>(gbase + (bars - base) + 256);          // [2][128]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    const int tiles = g.tiles_m * g.tiles_n;
    const int split = blockIdx.x / tiles, rem = blockIdx.x % tiles;
    const int m0 = (rem / g.tiles_n) * BM, n0 = (rem % g.tiles_n) * BN;
    const long long kb0 = (long long)split * g.per;
    const long long kb1 = (kb0 + g.per < g.g.nboxes) ? kb0 + g.per : g.g.nboxes;
    const long long nkb = kb1 - kb0;                                                    // >= 1 (host guarantees)
    const long long nseg = (nkb + RED_SEG - 1) / RED_SEG;

    // rows of the raw stages that a short TMA box (rb * nbx < 32) never writes must read as zero
    if (g.g.rb * g.g.nbx < BK) {
        float4 *z = reinterpret_cast<float4 *>(gbase);
        for (int i = threadIdx.x; i < RED_RAW_STAGES * RED_RAW_BYTES / 16; i += RED_NT) z[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        fence_proxy_async();
    }
    if (threadIdx.x == 0) {
        for (int s = 0; s < RED_RAW_STAGES; ++s) { mbar_init(bar_rfull(s), 1); mbar_init(bar_rempty(s), 256); }
        for (int s = 0; s < RED_OP_STAGES; ++s) { mbar_init(bar_ofull(s), 256); mbar_init(bar_oempty(s), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(bar_afull(a), 1); mbar_init(bar_aempty(a), 256); }
        fence_barrier_init();
    }
    if (warp == 17) tmem_alloc(tmem_slot, 512);            // columns [0,128) [128,256): main x 2; [256,384): small terms
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

    if (warp == 16) {
        if (elect_one()) {
            tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmB);
            const uint32_t box_bytes = (uint32_t)(g.g.rb * g.g.nbx * 128 * 4);
            for (long long i = 0; i < nkb; ++i) {
                const int s = (int)(i % RED_RAW_STAGES);
                const uint32_t ph = (uint32_t)((i / RED_RAW_STAGES) & 1);
                const long long box = kb0 + i;
                const int b0 = (int)(box / g.g.tpb) * g.g.nbx, t0 = (int)(box % g.g.tpb) * g.g.rb;
                mbar_wait(bar_rempty(s), ph ^ 1u);
                mbar_arrive_expect_tx(bar_rfull(s), 2 * box_bytes);
                tma_load_3d(raw0 + s * RED_RAW_BYTES, &tmA, bar_rfull(s), m0, t0, b0);
                tma_load_3d(raw0 + s * RED_RAW_BYTES + TILE_BYTES, &tmB, bar_rfull(s), n0, t0, b0);
            }
        }
    } else if (warp == 17) {
        if (elect_one()) {
            const uint32_t idesc = umma_idesc_tf32(BM, BN);
            for (long long i = 0; i < nkb; ++i) {
                const long long seg = i / RED_SEG;
                const int ab = (int)(seg & 1);
                const bool seg_first = (i % RED_SEG) == 0, seg_last = ((i + 1) % RED_SEG) == 0 || i + 1 == nkb;
                if (seg_first) {
                    mbar_wait(bar_aempty(ab), (uint32_t)(((seg >> 1) & 1) ^ 1));
                    tc_fence_after();
                }
                const int s = (int)(i % RED_OP_STAGES);
                const uint32_t ph = (uint32_t)((i / RED_OP_STAGES) & 1);
                mbar_wait(bar_ofull(s), ph);
                tc_fence_after();
                const uint32_t st = op0 + s * RED_OP_BYTES;
                issue_block_3x(tmem_base + ab * BN, tmem_base + 2 * BN, st, st + TILE_BYTES, st + 2 * TILE_BYTES, st + 3 * TILE_BYTES,
                               BK / 8, idesc, seg_first, i == 0, (i & 1) != 0);
                umma_commit(bar_oempty(s));
                if (seg_last) umma_commit(bar_afull(ab));
            }
        }
    } else if (warp < 8) {
        // ---------------- splitters (256 threads): raw [r][col] -> hi / lo [col][r] (K-major, 128-byte swizzle) -------
        const int col = threadIdx.x & 127, half = threadIdx.x >> 7;        // this thread: column `col`, r-quads 4*half .. 4*half+3
        const bool want_bias = g.pbias != nullptr && m0 == 0;
        float bsum = 0.f;
        for (long long i = 0; i < nkb; ++i) {
            const int rs = (int)(i % RED_RAW_STAGES), os = (int)(i % RED_OP_STAGES);
            const uint32_t rph = (uint32_t)((i / RED_RAW_STAGES) & 1), oph = (uint32_t)((i / RED_OP_STAGES) & 1);
            mbar_wait(bar_rfull(rs), rph);
            const float *rawA = reinterpret_cast<const float *>(gbase + rs * RED_RAW_BYTES);
            const float *rawB = rawA + TILE_BYTES / 4;
            float va[4][4], vb[4][4];
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int r = (4 * half + q) * 4 + e;
                    va[q][e] = rawA[r * 128 + col];
                    vb[q][e] = rawB[r * 128 + col];
                }
            if (want_bias)
#pragma unroll
                for (int q = 0; q < 4; ++q) bsum += (vb[q][0] + vb[q][1]) + (vb[q][2] + vb[q][3]);
            mbar_wait(bar_oempty(os), oph ^ 1u);
            uint8_t *op = gbase + (op0 - base) + os * RED_OP_BYTES;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int rq = 4 * half + q;
                const int off = col * 128 + ((rq ^ (col & 7)) << 4);
                float4 h, l;
                split4(make_float4(va[q][0], va[q][1], va[q][2], va[q][3]), h, l);
                *reinterpret_cast<float4 *>(op + off) = h;
                *reinterpret_cast<float4 *>(op + TILE_BYTES + off) = l;
                split4(make_float4(vb[q][0], vb[q][1], vb[q][2], vb[q][3]), h, l);
                *reinterpret_cast<float4 *>(op + 2 * TILE_BYTES + off) = h;
                *reinterpret_cast<float4 *>(op + 3 * TILE_BYTES + off) = l;
            }
            // Release the raw stage only now: the stores above take the loaded registers as operands, so every LDS of
            // this stage has completed.  (Arriving right after ISSUING the loads is a race: SYNCS.ARRIVE is not ordered
            // behind LDS that are still queued in the LSU, and the TMA refill can overtake them - measured, round 2.)
            mbar_arrive(bar_rempty(rs));
            fence_proxy_async();
            mbar_arrive(bar_ofull(os));
        }
        if (want_bias) {
            bias_red[half * 128 + col] = bsum;
            asm volatile("bar.sync 1, 256;" ::: "memory");                  // splitter warps only
            if (threadIdx.x < 128)
                g.pbias[(long long)split * g.N + n0 + threadIdx.x] = bias_red[threadIdx.x] + bias_red[128 + threadIdx.x];
        }
    } else {
        // ---------------- drain warps (256 threads): promote every finished TMEM segment into FP32 registers ----------
        const int dw = warp - 8;
        const int q = dw & 3, ch = dw >> 2;                                 // TMEM lane quarter (= warp % 4), 64-column half
        const uint32_t tl = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ch * 64);
        float acc[64];
#pragma unroll
        for (int j = 0; j < 64; ++j) acc[j] = 0.f;
        for (long long seg = 0; seg < nseg; ++seg) {
            const int ab = (int)(seg & 1);
            mbar_wait(bar_afull(ab), (uint32_t)((seg >> 1) & 1));
            tc_fence_after();
#pragma unroll
            for (int cc = 0; cc < 2; ++cc) {
                float v[32];
                tmem_ld32(tl + (uint32_t)(ab * BN + cc * 32), v);
#pragma unroll
                for (int j = 0; j < 32; ++j) acc[cc * 32 + j] += v[j];
            }
            tc_fence_before();
            mbar_arrive(bar_aempty(ab));
        }
        // the last segment's commit covers every MMA of the CTA: the small-term accumulator is complete too
        const int m = m0 + q * 32 + lane;
        float *prow = g.part + ((long long)split * g.M + m) * g.N + n0 + ch * 64;
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
            float v[32];
            tmem_ld32(tl + (uint32_t)(2 * BN + cc * 32), v);
            if (m < g.M) {
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    reinterpret_cast<float4 *>(prow + cc * 32)[j] =
                        make_float4(acc[cc * 32 + 4 * j] + v[4 * j], acc[cc * 32 + 4 * j + 1] + v[4 * j + 1],
                                    acc[cc * 32 + 4 * j + 2] + v[4 * j + 2], acc[cc * 32 + 4 * j + 3] + v[4 * j + 3]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 17) tmem_dealloc(tmem_base, 512);
}

// ---------------------------------------------------------------------------------------------------
// k_tc_red_ts: k_tc_red with the A operand in TMEM (tcgen05.mma "TS" form).  A row m of the 128 x 32 A tile is one TMEM
// lane: the four A-splitter warps (warp q owns lanes 32q..32q+31) read their column of the raw [32 r][128 m] tile, split it
// and write hi / lo with tcgen05.st; only B goes through shared memory (K-major SWIZZLE_128B, written by warps 4-7).
// Per k-block that removes 32 KB of operand-tile stores and 48 KB of MMA operand reads from the shared-memory port
// (224 -> 144 KB), which is what bounds k_tc_red, and frees shared memory for a deeper B ring.
// TMEM columns: [0,128) [128,256) main accumulators, [256,384) small terms, [384,512) two A stages of (hi 32 | lo 32).
// warps 0-3: A splitters; 4-7: B splitters (+ bias column sums); 8-15: drain; 16: TMA; 17: MMA issuer + TMEM allocator
// ---------------------------------------------------------------------------------------------------
constexpr int RTS_RAW_STAGES = 5, RTS_OP_STAGES = 2;
constexpr int RTS_OP_BYTES = 2 * TILE_BYTES;                 // B hi, B lo
constexpr int RTS_SMEM = RTS_RAW_STAGES * RED_RAW_BYTES + RTS_OP_STAGES * RTS_OP_BYTES + 1024 + 256;
static_assert(RTS_SMEM >= TMEM_EXCLUSIVE_SMEM, "TMEM co-residence rule");

__global__ void __launch_bounds__(RED_NT, 1)
k_tc_red_ts(const __grid_constant__ TcRedArgs g, const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t *gbase = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t raw0 = base, op0 = base + RTS_RAW_STAGES * RED_RAW_BYTES;
    const uint32_t bars = op0 + RTS_OP_STAGES * RTS_OP_BYTES;
    auto bar_rfull = [&](int s) { return bars + 8u * s; };
    auto bar_rempty = [&](int s) { return bars + 8u * (RTS_RAW_STAGES + s); };
    auto bar_ofull = [&](int s) { return bars + 8u * (2 * RTS_RAW_STAGES + s); };
    auto bar_oempty = [&](int s) { return bars + 8u * (2 * RTS_RAW_STAGES + RTS_OP_STAGES + s); };
    auto bar_afull = [&](int a) { return bars + 8u * (2 * RTS_RAW_STAGES + 2 * RTS_OP_STAGES + a); };
    auto bar_aempty = [&](int a) { return bars + 8u * (2 * RTS_RAW_STAGES + 2 * RTS_OP_STAGES + 2 + a); };
    const uint32_t tmem_slot = bars + 8u * (2 * RTS_RAW_STAGES + 2 * RTS_OP_STAGES + 4);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    const int tiles = g.tiles_m * g.tiles_n;
    const int split = blockIdx.x / tiles, rem = blockIdx.x % tiles;
    const int m0 = (rem / g.tiles_n) * BM, n0 = (rem % g.tiles_n) * BN;
    const long long kb0 = (long long)split * g.per;
    const long long kb1 = (kb0 + g.per < g.g.nboxes) ? kb0 + g.per : g.g.nboxes;
    const long long nkb = kb1 - kb0;
    const long long nseg = (nkb + RED_SEG - 1) / RED_SEG;

    if (g.g.rb * g.g.nbx < BK) {
        float4 *z = reinterpret_cast<float4 *>(gbase);
        for (int i = threadIdx.x; i < RTS_RAW_STAGES * RED_RAW_BYTES / 16; i += RED_NT) z[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        fence_proxy_async();
    }
    if (threadIdx.x == 0) {
        for (int s = 0; s < RTS_RAW_STAGES; ++s) { mbar_init(bar_rfull(s), 1); mbar_init(bar_rempty(s), 256); }
        for (int s = 0; s < RTS_OP_STAGES; ++s) { mbar_init(bar_ofull(s), 256); mbar_init(bar_oempty(s), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(bar_afull(a), 1); mbar_init(bar_aempty(a), 256); }
        fence_barrier_init();
    }
    if (warp == 17) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
    constexpr uint32_t A_COL0 = 3 * BN;                     // TMEM columns of the A stages

    if (warp == 16) {
        if (elect_one()) {
            tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmB);
            const uint32_t box_bytes = (uint32_t)(g.g.rb * g.g.nbx * 128 * 4);
            for (long long i = 0; i < nkb; ++i) {
                const int s = (int)(i % RTS_RAW_STAGES);
                const uint32_t ph = (uint32_t)((i / RTS_RAW_STAGES) & 1);
                const long long box = kb0 + i;
                const int b0 = (int)(box / g.g.tpb) * g.g.nbx, t0 = (int)(box % g.g.tpb) * g.g.rb;
                mbar_wait(bar_rempty(s), ph ^ 1u);
                mbar_arrive_expect_tx(bar_rfull(s), 2 * box_bytes);
                tma_load_3d(raw0 + s * RED_RAW_BYTES, &tmA, bar_rfull(s), m0, t0, b0);
                tma_load_3d(raw0 + s * RED_RAW_BYTES + TILE_BYTES, &tmB, bar_rfull(s), n0, t0, b0);
            }
        }
    } else if (warp == 17) {
        if (elect_one()) {
            const uint32_t idesc = umma_idesc_tf32(BM, BN);
#ifdef TC_PROBE
            long long w_aempty = 0, w_ofull = 0, t_issue = 0, tq;
            const long long t_begin = clock64();
#endif
            for (long long i = 0; i < nkb; ++i) {
                const long long seg = i / RED_SEG;
                const int ab = (int)(seg & 1);
                const bool seg_first = (i % RED_SEG) == 0, seg_last = ((i + 1) % RED_SEG) == 0 || i + 1 == nkb;
                if (seg_first) {
                    PROBE(w_aempty, mbar_wait(bar_aempty(ab), (uint32_t)(((seg >> 1) & 1) ^ 1)))
                    tc_fence_after();
                }
                const int s = (int)(i % RTS_OP_STAGES);
                const uint32_t ph = (uint32_t)((i / RTS_OP_STAGES) & 1);
                PROBE(w_ofull, mbar_wait(bar_ofull(s), ph))
                tc_fence_after();
#ifdef TC_PROBE
                const long long ti0 = clock64();
#endif
                const uint32_t st = op0 + s * RTS_OP_BYTES;
                const uint64_t dbh = umma_desc_sw128(st), dbl = umma_desc_sw128(st + TILE_BYTES);
                const uint32_t a_hi = tmem_base + A_COL0 + (uint32_t)s * 64u, a_lo = a_hi + 32u;
                const uint32_t d_main = tmem_base + ab * BN, d_small = tmem_base + 2 * BN;
                // grouped by accumulator, order alternating between k-blocks (see issue_block_3x)
#pragma unroll
                for (int pass = 0; pass < 2; ++pass) {
                    if ((pass == 0) == ((i & 1) != 0)) {
#pragma unroll
                        for (int ks = 0; ks < BK / 8; ++ks)
                            umma_tf32_ts(d_main, a_hi + ks * 8, dbh + (uint64_t)(ks * 2), idesc, (seg_first && ks == 0) ? 0u : 1u);
                    } else {
#pragma unroll
                        for (int ks = 0; ks < BK / 8; ++ks) {
                            umma_tf32_ts(d_small, a_lo + ks * 8, dbh + (uint64_t)(ks * 2), idesc, (i == 0 && ks == 0) ? 0u : 1u);
                            umma_tf32_ts(d_small, a_hi + ks * 8, dbl + (uint64_t)(ks * 2), idesc, 1u);
                        }
                    }
                }
                umma_commit(bar_oempty(s));
                if (seg_last) umma_commit(bar_afull(ab));
#ifdef TC_PROBE
                t_issue += clock64() - ti0;
#endif
            }
#ifdef TC_PROBE
            if (blockIdx.x == 3 && g.probe) {
                g.probe[0] = clock64() - t_begin; g.probe[1] = w_aempty; g.probe[2] = w_ofull; g.probe[3] = 0;
                g.probe[4] = 0; g.probe[5] = t_issue; g.probe[6] = nkb;
            }
#endif
        }
    } else if (warp < 4) {
        // ---------------- A splitters: column m of the raw tile -> TMEM lane m, hi / lo over 32 k columns ----------------
        const int m = warp * 32 + lane;
        for (long long i = 0; i < nkb; ++i) {
            const int rs = (int)(i % RTS_RAW_STAGES), os = (int)(i % RTS_OP_STAGES);
            const uint32_t rph = (uint32_t)((i / RTS_RAW_STAGES) & 1), oph = (uint32_t)((i / RTS_OP_STAGES) & 1);
            mbar_wait(bar_rfull(rs), rph);
            const float *rawA = reinterpret_cast<const float *>(gbase + rs * RED_RAW_BYTES);
            // split into registers BEFORE waiting for the operand stage: the ALU work overlaps the MMAs of the previous
            // k-block and only the TMEM stores stay on the oempty -> ofull critical path
            float hi[32], lo[32];
#pragma unroll
            for (int r = 0; r < 32; ++r) {
                const float x = rawA[r * 128 + m];
                hi[r] = tf32_rna(x);
                lo[r] = x - hi[r];                           // exact; kind::tf32 ignores the low 13 mantissa bits (<= 2^-21 |x|)
            }
            mbar_wait(bar_oempty(os), oph ^ 1u);             // the MMAs that read this A stage have completed
            tc_fence_after();
            const uint32_t ta = tmem_base + ((uint32_t)(warp * 32) << 16) + A_COL0 + (uint32_t)os * 64u;
            tmem_st32(ta, hi);
            tmem_st32(ta + 32, lo);
            tmem_wait_st();
            mbar_arrive(bar_rempty(rs));                     // after the values were consumed (see k_tc_red)
            tc_fence_before();
            mbar_arrive(bar_ofull(os));
        }
    } else if (warp < 8) {
        // ---------------- B splitters: raw [r][col] -> hi / lo [col][r] (K-major, 128-byte swizzle) + bias column sums ---------
        const int col = threadIdx.x - 128;
        const bool want_bias = g.pbias != nullptr && m0 == 0;
        float bsum = 0.f;
        for (long long i = 0; i < nkb; ++i) {
            const int rs = (int)(i % RTS_RAW_STAGES), os = (int)(i % RTS_OP_STAGES);
            const uint32_t rph = (uint32_t)((i / RTS_RAW_STAGES) & 1), oph = (uint32_t)((i / RTS_OP_STAGES) & 1);
            mbar_wait(bar_rfull(rs), rph);
            const float *rawB = reinterpret_cast<const float *>(gbase + rs * RED_RAW_BYTES + TILE_BYTES);
            float4 h[8], l[8];
#pragma unroll
            for (int rq = 0; rq < 8; ++rq) {
                const float4 vb = make_float4(rawB[(rq * 4 + 0) * 128 + col], rawB[(rq * 4 + 1) * 128 + col],
                                              rawB[(rq * 4 + 2) * 128 + col], rawB[(rq * 4 + 3) * 128 + col]);
                if (want_bias) bsum += (vb.x + vb.y) + (vb.z + vb.w);
                split4_trunc(vb, h[rq], l[rq]);
            }
            mbar_wait(bar_oempty(os), oph ^ 1u);
            uint8_t *op = gbase + (op0 - base) + os * RTS_OP_BYTES;
#pragma unroll
            for (int rq = 0; rq < 8; ++rq) {
                const int off = col * 128 + ((rq ^ (col & 7)) << 4);
                *reinterpret_cast<float4 *>(op + off) = h[rq];
                *reinterpret_cast<float4 *>(op + TILE_BYTES + off) = l[rq];
            }
            mbar_arrive(bar_rempty(rs));
            fence_proxy_async();
            mbar_arrive(bar_ofull(os));
        }
        if (want_bias) g.pbias[(long long)split * g.N + n0 + col] = bsum;
    } else {
        // ---------------- drain warps: promote every finished TMEM segment into FP32 registers (as in k_tc_red) ----------
        const int dw = warp - 8;
        const int q = dw & 3, ch = dw >> 2;
        const uint32_t tl = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ch * 64);
        float acc[64];
#pragma unroll
        for (int j = 0; j < 64; ++j) acc[j] = 0.f;
        for (long long seg = 0; seg < nseg; ++seg) {
            const int ab = (int)(seg & 1);
            mbar_wait(bar_afull(ab), (uint32_t)((seg >> 1) & 1));
            tc_fence_after();
#pragma unroll
            for (int cc = 0; cc < 2; ++cc) {
                float v[32];
                tmem_ld32(tl + (uint32_t)(ab * BN + cc * 32), v);
#pragma unroll
                for (int j = 0; j < 32; ++j) acc[cc * 32 + j] += v[j];
            }
            tc_fence_before();
            mbar_arrive(bar_aempty(ab));
        }
        const int m = m0 + q * 32 + lane;
        float *prow = g.part + ((long long)split * g.M + m) * g.N + n0 + ch * 64;
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
            float v[32];
            tmem_ld32(tl + (uint32_t)(2 * BN + cc * 32), v);
            if (m < g.M) {
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    reinterpret_cast<float4 *>(prow + cc * 32)[j] =
                        make_float4(acc[cc * 32 + 4 * j] + v[4 * j], acc[cc * 32 + 4 * j + 1] + v[4 * j + 1],
                                    acc[cc * 32 + 4 * j + 2] + v[4 * j + 2], acc[cc * 32 + 4 * j + 3] + v[4 * j + 3]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 17) tmem_dealloc(tmem_base, 512);
}

// ---------------------------------------------------------------------------------------------------
// host side: tensor maps and launchers.  Return 0 on success, a CUresult / cudaError_t code (> 0) otherwise,
// -1 when the shape cannot go through this path (caller falls back to the FFMA kernels)
// ---------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = []() -> EncodeTiledFn {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) != cudaSuccess || qr != cudaDriverEntryPointSuccess)
            return nullptr;
        return (EncodeTiledFn)p;
    }();
    return fn;
}

// 3-D FP32 map: dims (d0, d1, d2) elements, strides s1 / s2 in floats, box (b0, b1, b2)
inline int make_map(CUtensorMap *m, const float *p, long long d0, long long d1, long long d2, long long s1, long long s2,
                    int b0, int b1, int b2, bool swizzle128) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return 999;
    if (((uintptr_t)p & 15) || (s1 * 4) % 16 || (s2 * 4) % 16 || b0 > 256 || b1 > 256 || b2 > 256) return -1;
    cuuint64_t dims[3] = {(cuuint64_t)d0, (cuuint64_t)d1, (cuuint64_t)d2};
    cuuint64_t strides[2] = {(cuuint64_t)s1 * 4, (cuuint64_t)s2 * 4};
    cuuint32_t box[3] = {(cuuint32_t)b0, (cuuint32_t)b1, (cuuint32_t)b2};
    cuuint32_t es[3] = {1, 1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float *>(p), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : (int)r;
}

// ragged matrix -> (rpb, nb) with fully contiguous views collapsed to one batch entry
inline void rag_dims(long long rows, long long rpb, long long bstride, long long ld, long long *rpb_o, long long *nb_o, long long *bs_o) {
    if (rpb <= 0 || rpb >= rows || bstride == rpb * ld) { *rpb_o = rows; *nb_o = 1; *bs_o = rows * ld; }
    else { *rpb_o = rpb; *nb_o = (rows + rpb - 1) / rpb; *bs_o = bstride; }
}

inline bool tc_rows_ok(long long rows, int K, int N) { return rows >= 128 && K >= 8 && K % 4 == 0 && N % BN == 0; }
inline bool tc_red_ok(long long rows, int M, int N) { return rows >= 256 && M >= 64 && M % 4 == 0 && N % BN == 0; }

// C = A * Bt^T (+ biases); bt_hi / bt_lo: N x K pre-split copies of Bt
// 1 (default) = A operand from TMEM (k_tc_rows_ts) when K >= 128; 0 = both operands from shared memory (k_tc_rows).
// Measured on B200 (tools/tc_gemm_test, round 2, after the elect.sync issuer fix; rows 102 400 / 262 144):
//   K 256 N 1024: 0.353 vs 0.380 ms (152 vs 141 TFLOP/s)   K 1024 N 256: 0.278 vs 0.302 (193 vs 178)
//   K 256 N 4096: 3.414 vs 3.586 (161 vs 153)               K 40 N 1024: 0.222 vs 0.187 (epilogue-bound: shared-memory variant)
// Instrumented (-DTC_PROBE: clock64 around every wait of the MMA issuer): with K = 256 the issuer waits ~500 clk per k-block
// for the A operand stage -- the splitters' tcgen05.st queue behind the epilogue's tcgen05.ld (128 KB of accumulator reads per
// tile at 64 B/clk) -- and ~170 clk with K = 1024, where the MMAs run back to back (issue time = 12 x 65 clk per k-block).
inline int &tc_rows_variant() { static int v = 1; return v; }


inline int launch_tc_rows(long long rows, int rpb, const float *a, long long a_bstride, int K, const float *bt_hi,
                          const float *bt_lo, int N, const float *bias, const float *bias2, float *c, long long c_bstride,
                          int sms, cudaStream_t st, bool grad = false) {
    long long rp, nb, abs_, cbs, rp2, nb2;
    rag_dims(rows, rpb, a_bstride, K, &rp, &nb, &abs_);
    rag_dims(rows, rpb, c_bstride, N, &rp2, &nb2, &cbs);
    if (rp != rp2) { rp = rpb; nb = (rows + rpb - 1) / rpb; abs_ = a_bstride; cbs = c_bstride; }   // only one side contiguous
    TcRowsArgs g;
    g.g = make_ragbox(rp, nb, BM);
    g.K = K; g.N = N; g.tiles_n = N / BN;
    g.ntiles = g.g.nboxes * g.tiles_n;
    g.c = c; g.c_bstride = cbs; g.c_ld = N; g.bias = bias; g.bias2 = bias2;
#ifdef TC_PROBE
    g.probe = tc_probe_buf();
#endif
    CUtensorMap tmA, tmBh, tmBl;
    int rc = make_map(&tmA, a, K, rp, nb, K, abs_, BK, g.g.rb, g.g.nbx, true);
    if (rc) return rc;
    if ((rc = make_map(&tmBh, bt_hi, K, N, 1, K, (long long)N * K, BK, BN, 1, true))) return rc;
    if ((rc = make_map(&tmBl, bt_lo, K, N, 1, K, (long long)N * K, BK, BN, 1, true))) return rc;
    static bool attr = false;
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(k_tc_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, ROWS_SMEM);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_tc_rows_ts<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, RWT_SMEM);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_tc_rows_ts<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, RWT_SMEM);
        if (e != cudaSuccess) return (int)e;
        attr = true;
    }
    long long grid = g.ntiles < sms ? g.ntiles : sms;
    // short K: a tile is one or two k-blocks and the kernel is epilogue-bound; the single small-term accumulator of the TMEM
    // variant then stalls the MMAs (measured K = 40: 0.222 vs 0.187 ms)
    if (!tc_rows_variant() || K < 128) k_tc_rows<<<(unsigned)grid, ROWS_NT, ROWS_SMEM, st>>>(g, tmA, tmBh, tmBl);
    else if (grad) k_tc_rows_ts<true><<<(unsigned)grid, RWT_NT, RWT_SMEM, st>>>(g, tmA, tmBh, tmBl);
    else k_tc_rows_ts<false><<<(unsigned)grid, RWT_NT, RWT_SMEM, st>>>(g, tmA, tmBh, tmBl);
    return (int)cudaGetLastError();
}

// 1 (default) = A operand from TMEM (k_tc_red_ts); 0 = both operands from shared memory (k_tc_red).  Measured on B200
// (tools/tc_gemm_test, round 2, cfg3 / cfg5 shapes): shared-memory variant 164 / 174 / 176 TFLOP/s; A in TMEM with the same
// three raw stages 161 / 169 / 172 (the shared-memory port is not what binds these kernels); A in TMEM with the FIVE raw TMA
// stages its smaller operand ring makes room for: 169 / 177 / 183.  An L2 prefetch 8 k-blocks ahead of the TMA loads changed
// nothing.  ncu: tensor pipe active 49-51 %, which with cta_group::1 (M = 128) is half of what the unit can do; the kernels
// respond to pipeline depth (bytes in flight against the TMA latency), so a cta_group::2 pair (half of B per CTA, full-rate
// M = 256 MMAs) is the next step.
inline int &tc_red_variant() { static int v = 1; return v; }

inline int launch_tc_red(long long rows, int rpb, const float *a, long long a_bstride, int M, const float *b, long long b_bstride,
                         int N, float *part, float *pbias, int sms, int max_split, int *nsplit_out, cudaStream_t st) {
    long long rp, nb, abs_, rp2, nb2, bbs;
    rag_dims(rows, rpb, a_bstride, M, &rp, &nb, &abs_);
    rag_dims(rows, rpb, b_bstride, N, &rp2, &nb2, &bbs);
    if (rp != rp2) { rp = rpb; nb = (rows + rpb - 1) / rpb; abs_ = a_bstride; bbs = b_bstride; }
    TcRedArgs g;
    long long per = 0;
    RagBox gb = make_ragbox(rp, nb, BK);
    {
        // number of row splits: minimise waves x (k-blocks per split + a per-CTA prologue / epilogue cost)
        const long long tiles = (long long)((M + BM - 1) / BM) * (N / BN);
        long long best = 1;
        double best_cost = 1e300;
        for (long long s = 1; s <= max_split && s <= gb.nboxes; ++s) {
            const long long p = (gb.nboxes + s - 1) / s;
            const long long s_eff = (gb.nboxes + p - 1) / p;
            const long long waves = (tiles * s_eff + sms - 1) / sms;
            const double cost = (double)waves * ((double)p + 24.0);
            if (cost < best_cost) { best_cost = cost; best = s_eff; }
        }
        per = (gb.nboxes + best - 1) / best;
    }
    g.g = gb;
    g.M = M; g.N = N; g.tiles_m = (M + BM - 1) / BM; g.tiles_n = N / BN;
    g.per = per;
    g.nsplit = (int)((gb.nboxes + per - 1) / per);
    g.part = part; g.pbias = pbias;
#ifdef TC_PROBE
    g.probe = tc_probe_buf();
#endif
    CUtensorMap tmA, tmB;
    int rc = make_map(&tmA, a, M, rp, nb, M, abs_, 128, gb.rb, gb.nbx, false);
    if (rc) return rc;
    if ((rc = make_map(&tmB, b, N, rp, nb, N, bbs, 128, gb.rb, gb.nbx, false))) return rc;
    static bool attr = false;
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(k_tc_red, cudaFuncAttributeMaxDynamicSharedMemorySize, RED_SMEM);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_tc_red_ts, cudaFuncAttributeMaxDynamicSharedMemorySize, RTS_SMEM);
        if (e != cudaSuccess) return (int)e;
        attr = true;
    }
    const long long grid = (long long)g.tiles_m * g.tiles_n * g.nsplit;
    if (tc_red_variant()) k_tc_red_ts<<<(unsigned)grid, RED_NT, RTS_SMEM, st>>>(g, tmA, tmB);
    else k_tc_red<<<(unsigned)grid, RED_NT, RED_SMEM, st>>>(g, tmA, tmB);
    if (nsplit_out) *nsplit_out = g.nsplit;
    return (int)cudaGetLastError();
}

}  // namespace ttc
