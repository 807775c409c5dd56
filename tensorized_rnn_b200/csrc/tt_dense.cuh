// Dense LSTM / GRU baselines through the same engine (SURVEY.md 8f-3): the reference's `LSTM` / `GRU` modules
// (tensorized_rnn/lstm.py:7-41,44-135, gru.py:11-50,52-136) with dense nn.Linear weights, selected by
// `pmnist_test.py` without --tt and by `SpeakerEncoder(compression=None)`.
//
// A dense W_hh (G*H x H, 1 MiB at H = 256) does not fit one SM's shared memory, so this first version runs the
// recurrence as one tensor-core GEMM (tt_tc.cuh, 3xTF32; FFMA below 128 rows) + one fused gate kernel per timestep,
// with everything that does not depend on the recurrence batched over the whole sequence: the ih projection, dX, and
// both weight gradients (dW_ih = da^T X, dW_hh = du^T H_prev as reductions over all B*T rows).  A persistent
// cluster-split kernel (W_hh sliced over the CTAs of a cluster, h_t exchanged through DSMEM) is the follow-up.
//
// Gate kernels: one thread per (batch row, hidden unit), strided views into the (B, T, .) sequence buffers.
#pragma once
#include <cuda_runtime.h>
#include "tt_stage.cuh"

namespace ttd {

struct DenseStepArgs {
    long long B;
    int H;
    const float *a; long long lda;            // (B, G*H) view: W_ih x_t (+ b_ih)
    const float *u; long long ldu;            // (B, G*H) view: W_hh h_{t-1} (+ b_hh)
    const float *h_prev; long long ldhp;      // (B, H) view or null (zeros)
    const float *c_prev; long long ldcp;      // LSTM: (B, H) view or null (zeros)
    float *h; long long ldh;                  // forward: h_t view
    float *c; long long ldc;                  // forward: c_t view (LSTM)
    // backward
    const float *dout; long long lddo;        // (B, H) view of dOut[:, t, :] or null
    const float *dh_gemm;                     // (B, H) contiguous: du_{t+1} W_hh, or null
    const float *dh_direct;                   // (B, H) contiguous: direct term of step t+1 (GRU), or null
    const float *dh_T;                        // (B, H) contiguous: upstream gradient of the final state (t = T-1 only) or null
    float *da; long long ldda;                // written (may alias a)
    float *du; long long lddu;                // written (may alias u)
    float *dh_direct_out;                     // (B, H) contiguous: GRU dh * z, LSTM not written
    float *dc;                                // (B, H) contiguous: LSTM cell-state gradient carry (read and overwritten)
    const float *dc_T;                        // LSTM: upstream gradient of c_T (t = T-1 only) or null
    int first;                                // backward: 1 at t = T-1 (dc carry starts from dc_T / zero)
};

template <bool LSTM>
__global__ void __launch_bounds__(256) k_dense_cell_fwd(const DenseStepArgs p) {
    const long long n = p.B * p.H;
    const int H = p.H;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const long long b = e / H;
        const int h = (int)(e - b * H);
        const float *ar = p.a + b * p.lda, *ur = p.u + b * p.ldu;
        if (LSTM) {
            const float ig = tt_sigmoid(ar[h] + ur[h]);
            const float fg = tt_sigmoid(ar[H + h] + ur[H + h]);
            const float gg = tanhf(ar[2 * H + h] + ur[2 * H + h]);
            const float og = tt_sigmoid(ar[3 * H + h] + ur[3 * H + h]);
            const float cp = p.c_prev ? p.c_prev[b * p.ldcp + h] : 0.f;
            const float cn = fg * cp + ig * gg;
            p.c[b * p.ldc + h] = cn;
            p.h[b * p.ldh + h] = og * tanhf(cn);
        } else {
            const float rg = tt_sigmoid(ar[h] + ur[h]);
            const float zg = tt_sigmoid(ar[H + h] + ur[H + h]);
            const float ng = tanhf(ar[2 * H + h] + rg * ur[2 * H + h]);
            const float hp = p.h_prev ? p.h_prev[b * p.ldhp + h] : 0.f;
            p.h[b * p.ldh + h] = (1.0f - zg) * ng + zg * hp;
        }
    }
}

// analytic backward of one step (SURVEY.md 8a-10); gates recomputed from a, u (da / du may overwrite them in place:
// every thread reads all of its gate inputs before it writes)
template <bool LSTM>
__global__ void __launch_bounds__(256) k_dense_cell_bwd(const DenseStepArgs p) {
    const long long n = p.B * p.H;
    const int H = p.H;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const long long b = e / H;
        const int h = (int)(e - b * H);
        float dh = 0.f;
        if (p.dout) dh += p.dout[b * p.lddo + h];
        if (p.dh_gemm) dh += p.dh_gemm[e];
        if (p.dh_direct) dh += p.dh_direct[e];
        if (p.dh_T) dh += p.dh_T[e];
        const float *ar = p.a + b * p.lda, *ur = p.u + b * p.ldu;
        float *dar = p.da + b * p.ldda, *dur = p.du + b * p.lddu;
        if (LSTM) {
            const float ig = tt_sigmoid(ar[h] + ur[h]);
            const float fg = tt_sigmoid(ar[H + h] + ur[H + h]);
            const float gg = tanhf(ar[2 * H + h] + ur[2 * H + h]);
            const float og = tt_sigmoid(ar[3 * H + h] + ur[3 * H + h]);
            const float cp = p.c_prev ? p.c_prev[b * p.ldcp + h] : 0.f;
            const float cn = fg * cp + ig * gg;
            const float tc = tanhf(cn);
            float dcn = dh * og * (1.0f - tc * tc);
            if (p.first) { if (p.dc_T) dcn += p.dc_T[e]; }
            else dcn += p.dc[e];
            const float d0 = dcn * gg * ig * (1.0f - ig);
            const float d1 = dcn * cp * fg * (1.0f - fg);
            const float d2 = dcn * ig * (1.0f - gg * gg);
            const float d3 = dh * tc * og * (1.0f - og);
            dar[h] = d0; dar[H + h] = d1; dar[2 * H + h] = d2; dar[3 * H + h] = d3;
            if (dur != dar) { dur[h] = d0; dur[H + h] = d1; dur[2 * H + h] = d2; dur[3 * H + h] = d3; }
            p.dc[e] = dcn * fg;
        } else {
            const float un = ur[2 * H + h];
            const float rg = tt_sigmoid(ar[h] + ur[h]);
            const float zg = tt_sigmoid(ar[H + h] + ur[H + h]);
            const float ng = tanhf(ar[2 * H + h] + rg * un);
            const float hp = p.h_prev ? p.h_prev[b * p.ldhp + h] : 0.f;
            const float d_n = dh * (1.0f - zg) * (1.0f - ng * ng);
            const float d_z = dh * (hp - ng) * zg * (1.0f - zg);
            const float d_r = d_n * un * rg * (1.0f - rg);
            dar[h] = d_r; dar[H + h] = d_z; dar[2 * H + h] = d_n;
            dur[h] = d_r; dur[H + h] = d_z; dur[2 * H + h] = d_n * rg;
            p.dh_direct_out[e] = dh * zg;
        }
    }
}

// u[b, :] = bias (or zero): the hh pre-activation of the first step without an initial state
__global__ void __launch_bounds__(256) k_bias_rows(const float *__restrict__ bias, float *__restrict__ u, long long ldu, long long B,
                                                   int N) {
    const long long n = B * N;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const long long b = e / N;
        const int c = (int)(e - b * N);
        u[b * ldu + c] = bias ? bias[c] : 0.f;
    }
}

// part[s][n] = sum of m[r, n] over the rows of split s   (grid: ceil(N / 128) x nsplit, 128 threads = 128 columns)
__global__ void __launch_bounds__(128) k_colsum_part(const float *__restrict__ m, long long rows, int N, int nsplit,
                                                     float *__restrict__ part) {
    const int n = blockIdx.x * 128 + threadIdx.x, s = blockIdx.y;
    if (n >= N) return;
    const long long per = (rows + nsplit - 1) / nsplit;
    const long long r0 = s * per, r1 = (r0 + per < rows) ? r0 + per : rows;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    long long r = r0;
    for (; r + 3 < r1; r += 4) {
        a0 += m[r * N + n]; a1 += m[(r + 1) * N + n]; a2 += m[(r + 2) * N + n]; a3 += m[(r + 3) * N + n];
    }
    for (; r < r1; ++r) a0 += m[r * N + n];
    part[(long long)s * N + n] = (a0 + a1) + (a2 + a3);
}

// Input widths that are not a multiple of 4 (pixel-by-pixel MNIST: input_size = 1) cannot go through the float4 GEMM
// loaders; the projection is then a handful of multiply-adds per output and runs on these plain kernels.
// y[r, n] = sum_k x[r, k] W[n, k] (+ bias[n]);  x rows contiguous (rows x K), y rows contiguous (rows x N)
__global__ void __launch_bounds__(256) k_smallk_fwd(const float *__restrict__ x, const float *__restrict__ W,
                                                    const float *__restrict__ bias, float *__restrict__ y, long long rows, int K,
                                                    int N) {
    const long long n_el = rows * N;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n_el; e += (long long)gridDim.x * blockDim.x) {
        const long long r = e / N;
        const int n = (int)(e - r * N);
        float t = bias ? bias[n] : 0.f;
        for (int k = 0; k < K; ++k) t += x[r * K + k] * __ldg(W + (long long)n * K + k);
        y[e] = t;
    }
}
// part[s][n, k] = sum over the rows of split s of da[r, n] x[r, k]   (grid: ceil(N / 128) x nsplit x K)
__global__ void __launch_bounds__(128) k_smallk_dw_part(const float *__restrict__ da, const float *__restrict__ x, long long rows,
                                                        int N, int K, int nsplit, float *__restrict__ part) {
    const int n = blockIdx.x * 128 + threadIdx.x, s = blockIdx.y, k = blockIdx.z;
    if (n >= N) return;
    const long long per = (rows + nsplit - 1) / nsplit;
    const long long r0 = s * per, r1 = (r0 + per < rows) ? r0 + per : rows;
    float a0 = 0.f, a1 = 0.f;
    long long r = r0;
    for (; r + 1 < r1; r += 2) {
        a0 += da[r * N + n] * x[r * K + k];
        a1 += da[(r + 1) * N + n] * x[(r + 1) * K + k];
    }
    if (r < r1) a0 += da[r * N + n] * x[r * K + k];
    part[((long long)s * N + n) * K + k] = a0 + a1;
}

// Projected LSTM backward, step t: dh_t = dOut[:, t, :] + carry (du_{t+1} W_hh, or the upstream d_hT at t = T-1), P wide,
// written into the (B, T, P) buffer that the dm_t GEMM reads now and the dW_hr GEMM reads after the loop.  dout and
// carry may be null (zero); carry is (B, P) contiguous.  One CTA per batch row (grid-stride over rows), threads over j.
__global__ void __launch_bounds__(128) k_dense_proj_dh(const float *__restrict__ dout, long long lddo,
                                                       const float *__restrict__ carry, float *__restrict__ dh, long long lddh,
                                                       long long B, int P) {
    for (long long b = blockIdx.x; b < B; b += gridDim.x)
        for (int j = threadIdx.x; j < P; j += blockDim.x)
            dh[b * lddh + j] = (dout ? dout[b * lddo + j] : 0.f) + (carry ? carry[b * P + j] : 0.f);
}

// out[e] = a[e] + (b ? b[e] : 0)
__global__ void __launch_bounds__(256) k_add2(const float *__restrict__ a, const float *__restrict__ b, float *__restrict__ out,
                                              long long n) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x)
        out[e] = a[e] + (b ? b[e] : 0.f);
}

}  // namespace ttd
