// Utterance-level embeddings (DESIGN.md §4.21): the two memory-bound kernels around the one stack call of
// SpeakerEncoder.embed_utterances.
//
//   k_partials_gather        out[w, t, :] = frames[first[w] + t, :] for t < valid[w], 0 for valid[w] <= t < P.
//                            A window's frames are consecutive rows of the packed (total_frames, F) block, so window w
//                            is the contiguous span frames[first[w] * F, (first[w] + valid[w]) * F) followed by zeros.
//                            One CTA per window, grid-stride over windows; float4 when F % 4 == 0.  A pure copy.
//   k_segment_mean_norm_fwd  y[s] = m / ||m||, m = mean of rows off[s] .. off[s+1]-1 of x (R, E); inv_norm[s] = 1 / ||m||.
//   k_segment_mean_norm_bwd  dx[r] = (dy[s] - y[s] (y[s] . dy[s])) * inv_norm[s] / count_s for every row r of segment s.
//
// One CTA per segment, grid-stride over segments, one thread per column (strided when E > NT).  Every sum runs in a
// fixed order with no atomics: a column's rows in row order (accumulated in double, so that a segment of thousands of
// rows keeps the FP32 mean), the squared norm and the dot product through ge2e::block_sum.  A zero mean gives
// 0 * (1 / 0), as ttrnn_embed_forward does for a zero row.  The kernels trust the tables: win_first + win_valid <=
// total_frames and non-decreasing offsets are the caller's preconditions (include/ttrnn_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "tt_ge2e.cuh"

namespace utter {

constexpr int NT = ge2e::NT;

template <typename V>
__global__ void __launch_bounds__(NT) k_partials_gather(const V *__restrict__ frames, const int64_t *__restrict__ first,
                                                        const int32_t *__restrict__ valid, V *__restrict__ out, int64_t W,
                                                        int P, int Fv) {
    const int64_t per = (int64_t)P * Fv;
    for (int64_t w = blockIdx.x; w < W; w += gridDim.x) {
        const V *src = frames + first[w] * Fv;
        const int64_t nv = (int64_t)valid[w] * Fv;
        V *dst = out + w * per;
        for (int64_t i = threadIdx.x; i < per; i += NT) {
            V v = {};
            if (i < nv) v = src[i];
            dst[i] = v;
        }
    }
}

__global__ void __launch_bounds__(NT) k_segment_mean_norm_fwd(const float *__restrict__ x, const int64_t *__restrict__ off,
                                                              float *__restrict__ y, float *__restrict__ inv_norm,
                                                              int64_t n_seg, int E) {
    __shared__ float red[NT / 32];
    for (int64_t s = blockIdx.x; s < n_seg; s += gridDim.x) {
        const int64_t r0 = off[s], r1 = off[s + 1];
        const double cnt = (double)(r1 - r0);
        float *ys = y + s * E;
        float ss = 0.f;
        for (int e = threadIdx.x; e < E; e += NT) {
            double t = 0.0;
#pragma unroll 4
            for (int64_t r = r0; r < r1; ++r) t += (double)x[r * E + e];
            const float m = (float)(t / cnt);
            ys[e] = m;                                    // read back below by the same thread
            ss += m * m;
        }
        const float inv = 1.0f / sqrtf(ge2e::block_sum(ss, red));
        for (int e = threadIdx.x; e < E; e += NT) ys[e] *= inv;
        if (threadIdx.x == 0) inv_norm[s] = inv;
    }
}

__global__ void __launch_bounds__(NT) k_segment_mean_norm_bwd(const int64_t *__restrict__ off, const float *__restrict__ y,
                                                              const float *__restrict__ inv_norm, const float *__restrict__ dy,
                                                              float *__restrict__ dx, int64_t n_seg, int E) {
    __shared__ float red[NT / 32];
    for (int64_t s = blockIdx.x; s < n_seg; s += gridDim.x) {
        const int64_t r0 = off[s], r1 = off[s + 1];
        const float *ys = y + s * E, *dys = dy + s * E;
        float dot = 0.f;
        for (int e = threadIdx.x; e < E; e += NT) dot += ys[e] * dys[e];
        dot = ge2e::block_sum(dot, red);
        const float sc = inv_norm[s] / (float)(r1 - r0);
        for (int e = threadIdx.x; e < E; e += NT) {
            const float g = (dys[e] - ys[e] * dot) * sc;
            for (int64_t r = r0; r < r1; ++r) dx[r * E + e] = g;
        }
    }
}

inline unsigned grid_for(int64_t n, int sms) {
    const int64_t cap = (int64_t)sms * 8;
    return (unsigned)(n < cap ? n : cap);
}

}  // namespace utter
