// Variable-length sequences (DESIGN.md §4.22): the small kernels around the unchanged recurrent kernels that let a padded
// (B, T, .) batch with per-row lengths len_b run through one stack call.
//
// The recurrent kernels never see the lengths.  Every route that reads a materialised ih projection xg[b, t, :] adds it to
// the hh part before the gate nonlinearity, so overwriting the gate columns of each padded (b, t), t >= len_b, FREEZES the
// row there: LSTM i = -inf, f = +inf, g = o = 0 gives sigmoid(i) = 0 and sigmoid(f) = 1 exactly, so c_t = c_{t-1} bit for
// bit; GRU z = +inf, r = n = 0 gives h_t = 0 * n + 1 * h_{t-1}.  At a frozen step with no incoming gradient every gate
// delta is exactly 0, so dW_ih, dX and the core gradients take nothing from padded steps and d_cT (LSTM) / d_hT (GRU)
// reach step len_b - 1 unchanged.  Padded inputs must be finite (0 * NaN = NaN in dW_ih).
//
//   k_varlen_freeze   xg (B, tc, G*H) chunk whose first step is t0: the gate columns of padded (b, t0 + t) are overwritten;
//                     only padded positions are written.
//   k_varlen_last     dst[b, :] = src[b, len_b - 1, :] of a (B, T, W) block: the LSTM h_n of a layer (its kernel's h_T
//                     is the output of the last padded step, not of step len_b - 1).
//   k_varlen_mask     dst[b, t, :] = src[b, t, :] for t0 + t < len_b, 0 after (src NULL = zeros; dst may alias src: then
//                     only the padded rows are written), and dh[b, :] added at t0 + t = len_b - 1 unless dh is NULL: the
//                     gradient of an LSTM h_n enters as an output gradient, the recurrent kernel then gets d_hT = 0.
//   k_varlen_reverse_add / k_varlen_join_fwd / k_varlen_join_bwd: tt_bidir.cuh's moves with each row reversed over its own
//                     length, x'[b, t] = x[b, len_b - 1 - t] for t < len_b; positions t >= len_b are written as 0.
//
// Everything is grid-stride with 64-bit indexing, deterministic and memory-bound (each output takes at most one FP32 add).
// The two kernels that run per time chunk of every layer, freeze and mask, take one (b, t) row per CTA iteration and its
// columns across the threads: the padding test is made once per row, so a row that is not padded costs one load of len_b
// (no per-element index division).
// The lengths are trusted device data: 1 <= len_b <= T for every row is the caller's precondition (include/ttrnn_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

namespace varlen {

constexpr int NT = 256;

#define VL_LOOP(i, n) for (long long i = blockIdx.x * (long long)NT + threadIdx.x; i < (n); i += (long long)gridDim.x * NT)

// the frozen ih pre-activation of gate column j (gate j / H; LSTM i, f, g, o, GRU r, z, n)
__device__ __forceinline__ float frozen_gate(int gate, bool lstm) {
    if (lstm) return gate == 0 ? -CUDART_INF_F : gate == 1 ? CUDART_INF_F : 0.f;
    return gate == 1 ? CUDART_INF_F : 0.f;
}

// xg: (B, tc, GH) at batch stride ld; rows = B * tc
__global__ void __launch_bounds__(NT) k_varlen_freeze(float *__restrict__ xg, long long ld, const int32_t *__restrict__ len,
                                                      long long rows, int tc, int t0, int GH, int H, int lstm) {
    for (long long row = blockIdx.x; row < rows; row += gridDim.x) {
        const long long b = row / tc;
        const int t = (int)(row - b * tc);
        if (t0 + t < len[b]) continue;
        float *x = xg + b * ld + (long long)t * GH;
        for (int j = threadIdx.x; j < GH; j += NT) x[j] = frozen_gate(j / H, lstm != 0);
    }
}

// src (B, T, W) at batch stride ld; n = B * W
__global__ void __launch_bounds__(NT) k_varlen_last(const float *__restrict__ src, long long ld, const int32_t *__restrict__ len,
                                                    float *__restrict__ dst, long long n, int W) {
    VL_LOOP(i, n) {
        const long long b = i / W;
        const int j = (int)(i - b * W);
        dst[i] = src[b * ld + (long long)(len[b] - 1) * W + j];
    }
}

// src / dst (B, tn, F) at batch strides ld_src / ld_dst, first step t0, dh (B, F) or NULL; rows = B * tn
__global__ void __launch_bounds__(NT) k_varlen_mask(const float *src, long long ld_src, float *dst, long long ld_dst,
                                                    const int32_t *__restrict__ len, const float *__restrict__ dh,
                                                    long long rows, int tn, int t0, int F) {
    const bool in_place = src == dst && ld_src == ld_dst;
    for (long long row = blockIdx.x; row < rows; row += gridDim.x) {
        const long long b = row / tn;
        const int t = (int)(row - b * tn);
        const int lb = len[b];
        const long long o = (long long)t * F;
        float *y = dst + b * ld_dst + o;
        if (t0 + t >= lb) {
            for (int j = threadIdx.x; j < F; j += NT) y[j] = 0.f;
            continue;
        }
        const float *d = (dh && t0 + t == lb - 1) ? dh + b * F : nullptr;
        if (in_place && !d) continue;
        const float *x = src ? src + b * ld_src + o : nullptr;
        for (int j = threadIdx.x; j < F; j += NT) {
            const float v = x ? x[j] : 0.f;
            y[j] = d ? v + d[j] : v;
        }
    }
}

// the step of row b that time-reverses step t over the row's length, or -1 past it
__device__ __forceinline__ int rev_t(int t, int l) { return t < l ? l - 1 - t : -1; }

// y[b,t,:] = a[b,t,:] + r[b,len_b-1-t,:] for t < len_b, else 0; n = B * T * F
__global__ void __launch_bounds__(NT) k_varlen_reverse_add(const float *__restrict__ a, const float *__restrict__ r,
                                                           float *__restrict__ y, const int32_t *__restrict__ len, long long n,
                                                           int T, int F) {
    VL_LOOP(i, n) {
        const long long row = i / F;
        const int j = (int)(i - row * F);
        const long long b = row / T;
        const int tr = rev_t((int)(row - b * T), len[b]);
        float v = 0.f;
        if (tr >= 0) {
            if (a && r) v = a[i] + r[(b * T + tr) * F + j];
            else if (a) v = a[i];
            else if (r) v = r[(b * T + tr) * F + j];
        }
        y[i] = v;
    }
}

// y[b,t] = [f[b,t] | r[b,len_b-1-t]] and y_rev[b,len_b-1-t] = y[b,t] for t < len_b; zeros past the length; n = B * T * 2H
__global__ void __launch_bounds__(NT) k_varlen_join_fwd(const float *__restrict__ f, const float *__restrict__ r,
                                                        float *__restrict__ y, float *__restrict__ y_rev,
                                                        const int32_t *__restrict__ len, long long n, int T, int H) {
    const int W2 = 2 * H;
    VL_LOOP(i, n) {
        const long long row = i / W2;
        const int c = (int)(i - row * W2);
        const long long b = row / T;
        const int t = (int)(row - b * T), tr = rev_t(t, len[b]);
        if (tr < 0) {
            y[i] = 0.f;
            if (y_rev) y_rev[i] = 0.f;
            continue;
        }
        const float v = c < H ? f[row * H + c] : r[(b * T + tr) * H + (c - H)];
        y[i] = v;
        if (y_rev) y_rev[(b * T + tr) * W2 + c] = v;
    }
}

// d_f[b,t] = dy[b,t,:H] + dy_rev[b,len_b-1-t,:H], d_r[b,s] = dy[b,len_b-1-s,H:] + dy_rev[b,s,H:]; zeros past the length;
// n = B * T * H
__global__ void __launch_bounds__(NT) k_varlen_join_bwd(const float *__restrict__ dy, const float *__restrict__ dy_rev,
                                                        float *__restrict__ d_f, float *__restrict__ d_r,
                                                        const int32_t *__restrict__ len, long long n, int T, int H) {
    const int W2 = 2 * H;
    VL_LOOP(i, n) {
        const long long row = i / H;
        const int c = (int)(i - row * H);
        const long long b = row / T;
        const int tr = rev_t((int)(row - b * T), len[b]);
        float vf = 0.f, vr = 0.f;
        if (tr >= 0) {
            const long long rr = b * T + tr;
            if (dy && dy_rev) {
                vf = dy[row * W2 + c] + dy_rev[rr * W2 + c];
                vr = dy[rr * W2 + H + c] + dy_rev[row * W2 + H + c];
            } else if (dy) {
                vf = dy[row * W2 + c];
                vr = dy[rr * W2 + H + c];
            } else if (dy_rev) {
                vf = dy_rev[rr * W2 + c];
                vr = dy_rev[row * W2 + H + c];
            }
        }
        d_f[i] = vf;
        d_r[i] = vr;
    }
}

#undef VL_LOOP

// one CTA per (b, t) row, at most 16 per SM
inline unsigned grid_rows(long long rows, int sms) {
    const long long cap = (long long)sms * 16;
    return (unsigned)(rows < 1 ? 1 : rows < cap ? rows : cap);
}

inline unsigned grid_for(long long n, int sms) {
    const long long want = (n + NT - 1) / NT, cap = (long long)sms * 16;
    return (unsigned)(want < 1 ? 1 : want < cap ? want : cap);
}

}  // namespace varlen
