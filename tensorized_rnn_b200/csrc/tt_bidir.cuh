// Direction handling of bidirectional stacks (DESIGN.md §4.17).  The reverse direction of a layer runs the unchanged
// one-layer recurrence on its input reversed in time, so all a bidirectional stack needs around the recurrent kernels is
// moving (B, T, F) blocks with time reversed, plus the adjoint sums of those moves.  Everything here is memory-bound:
// one thread per float4 (or per float when the feature width is not a multiple of 4), grid-stride, 64-bit indexing.
//
//   k_reverse_add  y[b,t,:] = a[b,t,:] + r[b,T-1-t,:]           a or r may be NULL (= zero)
//   k_join_fwd     y[b,t,:H] = f[b,t,:],  y[b,t,H:] = r[b,T-1-t,:],  y_rev[b,T-1-t,:] = y[b,t,:]   (y_rev may be NULL)
//   k_join_bwd     d_f[b,t,:] = dy[b,t,:H] + dy_rev[b,T-1-t,:H]
//                  d_r[b,s,:] = dy[b,T-1-s,H:] + dy_rev[b,s,H:]   dy or dy_rev may be NULL (= zero)
//
// Each output element takes exactly one FP32 add (none when an operand is NULL), so a result equals the sum PyTorch
// would form of the same two operands bit for bit.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace bidir {

constexpr int NT = 256;

template <int V> struct Vec;
template <> struct Vec<1> { typedef float T; };
template <> struct Vec<4> { typedef float4 T; };

__device__ __forceinline__ float vadd(float a, float b) { return a + b; }
__device__ __forceinline__ float4 vadd(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
template <typename T> __device__ __forceinline__ T vzero();
template <> __device__ __forceinline__ float vzero<float>() { return 0.f; }
template <> __device__ __forceinline__ float4 vzero<float4>() { return make_float4(0.f, 0.f, 0.f, 0.f); }

// row index (b * T + t) of the same batch row at time T-1-t
__device__ __forceinline__ long long rev_row(long long row, int T) {
    const long long b = row / T;
    return b * T + (T - 1) - (row - b * T);
}

// n = B * T * (F / V) vectors; fv = F / V
template <int V>
__global__ void __launch_bounds__(NT) k_reverse_add(const float *__restrict__ a, const float *__restrict__ r,
                                                    float *__restrict__ y, long long n, int T, int fv) {
    typedef typename Vec<V>::T VT;
    const VT *av = reinterpret_cast<const VT *>(a);
    const VT *rv = reinterpret_cast<const VT *>(r);
    VT *yv = reinterpret_cast<VT *>(y);
    for (long long i = blockIdx.x * (long long)NT + threadIdx.x; i < n; i += (long long)gridDim.x * NT) {
        const long long row = i / fv, c = i - row * fv;
        VT v;
        if (av && rv) v = vadd(av[i], rv[rev_row(row, T) * fv + c]);
        else if (av) v = av[i];
        else if (rv) v = rv[rev_row(row, T) * fv + c];
        else v = vzero<VT>();
        yv[i] = v;
    }
}

// n = B * T * (2H / V) vectors of y; hv = H / V
template <int V>
__global__ void __launch_bounds__(NT) k_join_fwd(const float *__restrict__ f, const float *__restrict__ r,
                                                 float *__restrict__ y, float *__restrict__ y_rev, long long n, int T,
                                                 int hv) {
    typedef typename Vec<V>::T VT;
    const VT *fv = reinterpret_cast<const VT *>(f);
    const VT *rv = reinterpret_cast<const VT *>(r);
    VT *yv = reinterpret_cast<VT *>(y);
    VT *yr = reinterpret_cast<VT *>(y_rev);
    const int wv = 2 * hv;
    for (long long i = blockIdx.x * (long long)NT + threadIdx.x; i < n; i += (long long)gridDim.x * NT) {
        const long long row = i / wv;
        const int c = (int)(i - row * wv);
        const long long rr = rev_row(row, T);
        const VT v = c < hv ? fv[row * hv + c] : rv[rr * hv + (c - hv)];
        yv[i] = v;
        if (yr) yr[rr * wv + c] = v;
    }
}

// n = B * T * (H / V) vectors of each of d_f and d_r; hv = H / V
template <int V>
__global__ void __launch_bounds__(NT) k_join_bwd(const float *__restrict__ dy, const float *__restrict__ dy_rev,
                                                 float *__restrict__ d_f, float *__restrict__ d_r, long long n, int T,
                                                 int hv) {
    typedef typename Vec<V>::T VT;
    const VT *g = reinterpret_cast<const VT *>(dy);
    const VT *gr = reinterpret_cast<const VT *>(dy_rev);
    VT *df = reinterpret_cast<VT *>(d_f);
    VT *dr = reinterpret_cast<VT *>(d_r);
    const int wv = 2 * hv;
    for (long long i = blockIdx.x * (long long)NT + threadIdx.x; i < n; i += (long long)gridDim.x * NT) {
        const long long row = i / hv;
        const int c = (int)(i - row * hv);
        const long long rr = rev_row(row, T);
        VT vf, vr;
        if (g && gr) {
            vf = vadd(g[row * wv + c], gr[rr * wv + c]);
            vr = vadd(g[rr * wv + hv + c], gr[row * wv + hv + c]);
        } else if (g) {
            vf = g[row * wv + c];
            vr = g[rr * wv + hv + c];
        } else if (gr) {
            vf = gr[rr * wv + c];
            vr = gr[row * wv + hv + c];
        } else {
            vf = vr = vzero<VT>();
        }
        df[i] = vf;
        dr[i] = vr;
    }
}

inline unsigned grid_for(long long n, int sms) {
    const long long want = (n + NT - 1) / NT, cap = (long long)sms * 16;
    return (unsigned)(want < cap ? want : cap);
}

}  // namespace bidir
