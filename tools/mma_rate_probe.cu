// Micro-benchmark: cycles per tcgen05.mma kind::tf32 dispatch on sm_100a, for the issue patterns of csrc/tt_tc.cuh,
// and the per-step round trip of the tensor-core stage 0 of the contracted BPTT kernel (tts::TcStage0).
// One CTA per SM, operands are whatever shared memory / TMEM holds (timing only).  Build:
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 --expt-relaxed-constexpr tools/mma_rate_probe.cu -o tools/mma_rate_probe
#include <cstdio>
#include <cstdlib>

#include "../tensorized_rnn_b200/csrc/tt_plan.h"
#include "../tensorized_rnn_b200/csrc/tt_static.cuh"
#include "../tensorized_rnn_b200/csrc/tt_tc.cuh"

using namespace ttc;

// mode 0: SS form, one accumulator          mode 1: TS form, one accumulator
// mode 2: TS form, the 3xTF32 pattern (small, small, main) of k_tc_red_ts, k-slices walking through a 128-byte row
// mode 3: SS form, 3xTF32 pattern (k_tc_rows)
// N = 128 or 256
__global__ void __launch_bounds__(256, 1) k_probe(int mode, int N, int iters, long long *out, int bg) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar = base + 6 * TILE_BYTES, slot = bar + 32;
    __shared__ int done;
    if (threadIdx.x == 0) { done = 0; mbar_init(bar, 1); mbar_init(bar + 16, 1); fence_barrier_init(); }
    if (threadIdx.x < 32) tmem_alloc(slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tb;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tb) : "r"(slot));
    if (bg & 4) {                                            // random operands instead of whatever the memories held (zeros)
        float *f = reinterpret_cast<float *>(smem_raw + (base - smem_u32(smem_raw)));
        uint32_t x = 1234567u + threadIdx.x * 7919u + blockIdx.x;
        for (int i = threadIdx.x; i < 6 * TILE_BYTES / 4; i += blockDim.x) {
            x = x * 1664525u + 1013904223u;
            f[i] = (float)(x >> 8) * (1.0f / 8388608.0f) - 1.0f;
        }
        fence_proxy_async();
        if (threadIdx.x < 128) {
            float v[32];
            for (int j = 0; j < 32; ++j) { x = x * 1664525u + 1013904223u; v[j] = (float)(x >> 8) * (1.0f / 8388608.0f) - 1.0f; }
            const uint32_t ta = tb + ((uint32_t)((threadIdx.x >> 5) & 3) * 32 << 16);
            for (int c = 0; c < 512; c += 32) tmem_st32(ta + c, v);
            tmem_wait_st();
        }
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
    }
    if (threadIdx.x == 0) {
        const uint32_t idesc = umma_idesc_tf32(128, N);
        const uint64_t da = umma_desc_sw128(base), da2 = umma_desc_sw128(base + TILE_BYTES);
        const uint64_t db = umma_desc_sw128(base + 2 * TILE_BYTES), db2 = umma_desc_sw128(base + 4 * TILE_BYTES);
        const uint32_t a_t = tb + 384, d0 = tb, d1 = tb + (N == 128 ? 128 : 256);
        const long long t0 = clock64();
        for (int i = 0; i < iters; ++i) {
            if (mode == 4) {                                 // TS, grouped by accumulator, order alternating per k-block
                for (int pass = 0; pass < 2; ++pass) {
                    if ((pass == 0) == ((i & 1) != 0)) {
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks) umma_tf32_ts(d0, a_t + ks * 8, db + (uint64_t)(ks * 2), idesc, 1u);
                    } else {
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks) {
                            umma_tf32_ts(d1, a_t + 32 + ks * 8, db + (uint64_t)(ks * 2), idesc, 1u);
                            umma_tf32_ts(d1, a_t + ks * 8, db2 + (uint64_t)(ks * 2), idesc, 1u);
                        }
                    }
                }
                continue;
            }
            if (mode == 5) {                                 // TS, accumulator alternating on every MMA
#pragma unroll
                for (int j = 0; j < 12; ++j) umma_tf32_ts((j & 1) ? d1 : d0, a_t + (j & 3) * 8, db + (uint64_t)((j & 3) * 2), idesc, 1u);
                continue;
            }
            if (mode == 6) {                                 // TS, one accumulator, one fixed k-slice (no operand address change)
#pragma unroll
                for (int j = 0; j < 12; ++j) umma_tf32_ts(d0, a_t, db, idesc, 1u);
                continue;
            }
            if (mode == 7) {                                 // TS, one accumulator, 12 MMAs then a commit (as the kernels do per k-block)
#pragma unroll
                for (int j = 0; j < 12; ++j) umma_tf32_ts(d0, a_t + (j & 3) * 8, db + (uint64_t)((j & 3) * 2), idesc, 1u);
                umma_commit(bar + 16);
                continue;
            }
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
                const uint64_t o = (uint64_t)(ks * 2);
                if (mode == 0) {
                    umma_tf32(d0, da + o, db + o, idesc, 1u);
                    umma_tf32(d0, da2 + o, db + o, idesc, 1u);
                    umma_tf32(d0, da + o, db2 + o, idesc, 1u);
                } else if (mode == 1) {
                    umma_tf32_ts(d0, a_t + ks * 8, db + o, idesc, 1u);
                    umma_tf32_ts(d0, a_t + 32 + ks * 8, db + o, idesc, 1u);
                    umma_tf32_ts(d0, a_t + ks * 8, db2 + o, idesc, 1u);
                } else if (mode == 2) {
                    umma_tf32_ts(d1, a_t + 32 + ks * 8, db + o, idesc, 1u);
                    umma_tf32_ts(d1, a_t + ks * 8, db2 + o, idesc, 1u);
                    umma_tf32_ts(d0, a_t + ks * 8, db + o, idesc, 1u);
                } else {
                    umma_tf32(d1, da2 + o, db + o, idesc, 1u);
                    umma_tf32(d1, da + o, db2 + o, idesc, 1u);
                    umma_tf32(d0, da + o, db + o, idesc, 1u);
                }
            }
        }
        umma_commit(bar);
        mbar_wait(bar, 0);
        const long long t1 = clock64();
        if (blockIdx.x == 0) out[0] = t1 - t0;
    }
    // background traffic while thread 0 issues: bg & 1 = warps 1-3 stream LDS.128 / STS.128 over 32 KB of shared memory,
    // bg & 2 = warps 4-7 keep writing 64 TMEM columns (tcgen05.st, as the A splitters of tt_tc.cuh do)
    if (threadIdx.x == 0) done = 1;
    if ((bg & 1) && threadIdx.x >= 32 && threadIdx.x < 128) {
        float4 *p4 = reinterpret_cast<float4 *>(smem_raw + (base - smem_u32(smem_raw)) + 6 * TILE_BYTES + 1024);
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        while (*(volatile int *)&done == 0) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                float4 v = p4[(threadIdx.x - 32) + 96 * j];
                acc.x += v.x;
                p4[(threadIdx.x - 32) + 96 * j] = acc;
            }
        }
        if (acc.x == 123.f) out[1] = 1;
    }
    if ((bg & 2) && threadIdx.x >= 128) {
        float v[32];
        for (int j = 0; j < 32; ++j) v[j] = (float)j;
        const uint32_t ta = tb + ((uint32_t)((threadIdx.x >> 5) & 3) * 32 << 16) + 256;
        while (*(volatile int *)&done == 0) {
            tmem_st32(ta, v);
            tmem_st32(ta + 32, v);
            tmem_wait_st();
        }
    }
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tmem_dealloc(tb, 512);
}

// Round trip of one step of the tensor-core stage 0 at R rows per CTA, as k_rnn_bwd_s runs it: every thread writes the
// hi / lo parts of its R gate-gradient chunks into the B buffers -> proxy fence + barrier -> 48 MMAs with A from TMEM ->
// commit -> mbarrier wait -> tcgen05.ld of 2 x 16R columns per thread -> stores into the X_0 slot -> barrier.
struct HH_d3r8 {
    static constexpr int D = 3, G = 4;
    static constexpr int J[7] = {4, 8, 8}, I[7] = {8, 8, 16}, RK[7] = {1, 8, 8, 1};
};
template <int R>
__global__ void __launch_bounds__(256, 1) k_step_probe(const float *cores, int steps, long long *out) {
    using S = tts::Merge01<HH_d3r8>;
    using TC0 = tts::TcStage0<S, R>;
    using T0 = tts::St<S, 0>;
    extern __shared__ __align__(16) float smem[];
    const int tid = threadIdx.x;
    float *x0 = smem;
    const uint32_t hi = (smem_u32(smem + R * T0::BS) + 1023u) & ~1023u, lo = hi + TC0::BUF_BYTES;
    const uint32_t bar = lo + TC0::BUF_BYTES, slot = bar + 8;
    char *hi_p = reinterpret_cast<char *>(smem) + (hi - smem_u32(smem)), *lo_p = hi_p + TC0::BUF_BYTES;
    if (tid == 0) { mbar_init(bar, 1); fence_barrier_init(); }
    if (tid < 32) tmem_alloc(slot, TC0::TCOLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tb = *reinterpret_cast<volatile uint32_t *>(reinterpret_cast<char *>(smem) + (slot - smem_u32(smem)));
    TC0::stage_a(cores, tb, tid);
    tc_fence_before();
    __syncthreads();
    const int mr = tid % T0::Mrow, i0p = tid / T0::Mrow;          // the hidden unit of the gate phase (one per thread)
    uint32_t phase = 0;
    const long long t0 = clock64();
    for (int t = 0; t < steps; ++t) {
#pragma unroll
        for (int b = 0; b < R; ++b) {
            const float v = x0[b * T0::BS + T0::roff(mr) + tid] * 0.5f + (float)(t + b);
            float4 h, l;
            split4_trunc(make_float4(v, v + 1.f, v + 2.f, v + 3.f), h, l);
            const uint32_t off = TC0::b_off(b * T0::Mrow + mr, i0p * 4);
            *reinterpret_cast<float4 *>(hi_p + off) = h;
            *reinterpret_cast<float4 *>(lo_p + off) = l;
        }
        fence_proxy_async();
        __syncthreads();
        if (tid < 32) {
            tc_fence_after();
            if (elect_one()) TC0::issue(tb, hi, lo, bar);
            __syncwarp();
        }
        mbar_wait(bar, phase);
        phase ^= 1u;
        tc_fence_after();
        TC0::drain(tb, x0, tid);
        tc_fence_before();
        __syncthreads();
    }
    const long long t1 = clock64();
    if (tid == 0) out[blockIdx.x] = t1 - t0;
    if (tid < 32) tmem_dealloc(tb, TC0::TCOLS);
}

template <int R>
void step_probe(const float *cores, long long *d) {
    using S = tts::Merge01<HH_d3r8>;
    static_assert(R * tts::St<S, 0>::BS * 4 + tts::TcStage0<S, R>::SMEM_BYTES <= ttc::TMEM_EXCLUSIVE_SMEM, "probe smem");
    cudaFuncSetAttribute(k_step_probe<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, ttc::TMEM_EXCLUSIVE_SMEM);
    const int steps = 160, reps = 20;
    k_step_probe<R><<<148, 256, ttc::TMEM_EXCLUSIVE_SMEM>>>(cores, steps, d);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    cudaEventRecord(e0);
    for (int i = 0; i < reps; ++i) k_step_probe<R><<<148, 256, ttc::TMEM_EXCLUSIVE_SMEM>>>(cores, steps, d);
    cudaEventRecord(e1);
    cudaError_t e = cudaDeviceSynchronize();
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    long long c[148];
    cudaMemcpy(c, d, sizeof(c), cudaMemcpyDeviceToHost);
    long long cmax = 0;
    double csum = 0;
    for (int i = 0; i < 148; ++i) { csum += c[i]; if (c[i] > cmax) cmax = c[i]; }
    printf("stage-0 round trip R=%d (N=%d, 148 CTAs, %d steps): %s  %.0f clk per step (mean over CTAs, max %.0f);  "
           "%.3f us per step (launch time / steps, incl. TMEM set-up)\n",
           R, 16 * R, steps, cudaGetErrorString(e), csum / 148 / steps, (double)cmax / steps, 1e3 * ms / reps / steps);
}

int main(int argc, char **argv) {
    long long *d;
    cudaMalloc(&d, 148 * 8);
    if (argc > 1 && argv[1][0] == 's') {                     // "step": the stage-0 round trip only
        float *cores;
        const int n = tts::core_floats<HH_d3r8>();
        cudaMalloc(&cores, n * 4);
        cudaMemset(cores, 0, n * 4);
        step_probe<1>(cores, d);
        step_probe<2>(cores, d);
        step_probe<3>(cores, d);
        step_probe<4>(cores, d);
        return 0;
    }
    const int smem = 6 * TILE_BYTES + 2048 + 96 * 16 * 16 + 1024;
    cudaFuncSetAttribute(k_probe, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    const int iters = 2000;
    for (int N : {128, 256})
        for (int mode = 0; mode < 8; ++mode) {
            if (N == 256 && mode >= 2) continue;             // two 256-column accumulators + the A columns do not fit
            for (int bg : {0, 4, 7}) {
                if (bg && mode != 1 && mode != 2 && mode != 4 && mode != 0) continue;
                k_probe<<<148, 256, smem>>>(mode, N, iters, d, bg);
                cudaError_t e = cudaDeviceSynchronize();
                long long c = 0;
                cudaMemcpy(&c, d, 8, cudaMemcpyDeviceToHost);
                printf("N=%d mode=%d bg=%d : %s  %.1f clk per MMA\n", N, mode, bg, cudaGetErrorString(e), (double)c / (iters * 12.0));
            }
        }
    return 0;
}
