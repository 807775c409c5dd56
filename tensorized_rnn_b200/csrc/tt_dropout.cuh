// Inter-layer dropout of multi-layer stacks (DESIGN.md §4.18): y = x * mask / (1 - p) between two layer passes, with the
// mask a pure function of (seed, offset, boundary k, global batch row b, t, feature j), so that it is regenerated, not
// stored, by the backward, and does not depend on row groups, time chunks, rows per CTA or streams.
//
// Mask of element e = (b * T + t) * F + j of boundary k (F = the width of the layer output, H or 2H):
//   Philox4x32-10 (curand_philox4x32_x.h), key = (lo32(seed), hi32(seed)),
//   counter = (lo32(e / 4), hi32(e / 4) | k << 16, lo32(offset), hi32(offset)),
//   word = output word e % 4;  keep when word < thr, thr = floor((1 - p) * 2^32) (p = 0: always, p = 1: never).
// One Philox call serves four consecutive elements, so the float4 path (F % 4 == 0) draws once per vector.
//
//   k_dropout   v = x[b,t,:] (+ xr[b,T-1-t,:] when xr is given);  v = keep ? v * scale : 0
//               y[b,t,:] = v;  yr[b,T-1-t,:] = v when yr is given
// y may alias x (in place); xr and yr must not alias x or y.  Memory-bound: one thread per float4 (or float),
// grid-stride, 64-bit indexing, as the kernels of tt_bidir.cuh.
#pragma once
#include <cuda_runtime.h>
#include <curand_philox4x32_x.h>
#include <stdint.h>

namespace ttdrop {

constexpr int NT = 256;

struct Mask {
    uint64_t seed, offset;
    unsigned long long thr;     // keep when the 32-bit word is below thr (0 .. 2^32)
    long long row0;             // global batch row of local row 0
    unsigned boundary;          // k: the output of layer k
    float scale;                // 1 / (1 - p); 0 when p = 1
};

// the four mask words of elements 4q .. 4q+3 of boundary k
__device__ __forceinline__ uint4 mask_words(const Mask &m, unsigned long long q) {
    const uint4 c = make_uint4((unsigned)q, (unsigned)(q >> 32) | (m.boundary << 16), (unsigned)m.offset,
                               (unsigned)(m.offset >> 32));
    return curand_Philox4x32_10(c, make_uint2((unsigned)m.seed, (unsigned)(m.seed >> 32)));
}

// keep / drop of one element of boundary m.boundary at global element index e
__device__ __forceinline__ bool keep_element(const Mask &m, unsigned long long e) {
    const uint4 w = mask_words(m, e >> 2);
    const unsigned r = e & 3;
    const unsigned v = r == 0 ? w.x : (r == 1 ? w.y : (r == 2 ? w.z : w.w));
    return (unsigned long long)v < m.thr;
}

__device__ __forceinline__ long long rev_row(long long row, int T) {
    const long long b = row / T;
    return b * T + (T - 1) - (row - b * T);
}

// n = B * T * F scalars; F = feature width
__global__ void __launch_bounds__(NT) k_dropout_1(const float *x, const float *__restrict__ xr, float *y,
                                                  float *__restrict__ yr, long long n, int T, int F, Mask m) {
    const long long base = m.row0 * (long long)T * F;          // global index of local element 0
    for (long long i = blockIdx.x * (long long)NT + threadIdx.x; i < n; i += (long long)gridDim.x * NT) {
        const long long row = i / F, c = i - row * F;
        const long long ri = rev_row(row, T) * F + c;
        float v = x[i];
        if (xr) v += xr[ri];
        v = keep_element(m, (unsigned long long)(base + i)) ? v * m.scale : 0.f;
        y[i] = v;
        if (yr) yr[ri] = v;
    }
}

// n = B * T * F / 4 vectors; fv = F / 4 (F % 4 == 0, 16-byte aligned operands)
__global__ void __launch_bounds__(NT) k_dropout_4(const float *x, const float *__restrict__ xr, float *y,
                                                  float *__restrict__ yr, long long n, int T, int fv, Mask m) {
    const float4 *xv = reinterpret_cast<const float4 *>(x);
    const float4 *xrv = reinterpret_cast<const float4 *>(xr);
    float4 *yv = reinterpret_cast<float4 *>(y);
    float4 *yrv = reinterpret_cast<float4 *>(yr);
    const long long base = m.row0 * (long long)T * fv;         // global vector index of local vector 0
    for (long long i = blockIdx.x * (long long)NT + threadIdx.x; i < n; i += (long long)gridDim.x * NT) {
        const long long row = i / fv, c = i - row * fv;
        const long long ri = rev_row(row, T) * fv + c;
        float4 v = xv[i];
        if (xrv) {
            const float4 r = xrv[ri];
            v = make_float4(v.x + r.x, v.y + r.y, v.z + r.z, v.w + r.w);
        }
        const uint4 w = mask_words(m, (unsigned long long)(base + i));
        v.x = (unsigned long long)w.x < m.thr ? v.x * m.scale : 0.f;
        v.y = (unsigned long long)w.y < m.thr ? v.y * m.scale : 0.f;
        v.z = (unsigned long long)w.z < m.thr ? v.z * m.scale : 0.f;
        v.w = (unsigned long long)w.w < m.thr ? v.w * m.scale : 0.f;
        yv[i] = v;
        if (yrv) yrv[ri] = v;
    }
}

inline unsigned grid_for(long long n, int sms) {
    const long long want = (n + NT - 1) / NT, cap = (long long)sms * 16;
    return (unsigned)(want < cap ? want : cap);
}

}  // namespace ttdrop
