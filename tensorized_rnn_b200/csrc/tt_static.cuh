// Statically specialised TT chain engine (sm_100a): every mode size, rank, row count and thread
// mapping is a compile-time constant, so index arithmetic folds away, the k-loops unroll and the
// gate math fuses into the epilogue of the last contraction stage.  Instantiated for the shapes
// registered in tt_static_inst.cu; every other shape runs on the runtime-shape kernels of
// tt_kernels.cuh (same maths, same C ABI).
//
// Restrictions of the static path (checked by static_assert / by the registry):
//   inner ranks r_1..r_{d-1} multiples of 4, every K_k = j_k * r_{k+1} a multiple of 4,
//   gates aligned with the first output mode (i_0 % G == 0), final-stage tiles <= one per thread.
#pragma once
#include <cuda_runtime.h>
#include <type_traits>
#include "tt_plan.h"

namespace tts {

constexpr int NTHR = 256;

constexpr int cpad(int k) { return (k % 4 != 0) ? k : (((k / 4) % 2 == 1) ? k : k + 4); }
constexpr int cr4(int v) { return (v + 3) & ~3; }
constexpr int cmin(int a, int b) { return a < b ? a : b; }
constexpr int cmax(int a, int b) { return a > b ? a : b; }
constexpr int p2floor(int v) { int p = 1; while (p * 2 <= v) p *= 2; return p; }
// largest power of two <= want that divides n (>= 1)
constexpr int p2div(int n, int want) {
    int p = p2floor(cmax(want, 1));
    while (p > 1 && n % p != 0) p /= 2;
    return p;
}

#define TTS_DEV __device__ __forceinline__
// k-loops over groups of four: fully unrolled up to 8 groups (no loop-carried register shuffles), else by 4
constexpr int unroll_of(int groups) { return groups <= 8 ? groups : 4; }

TTS_DEV void cp_async16(float *smem_dst, const float *gsrc) {
    unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gsrc));
}
TTS_DEV void cp_async4(float *smem_dst, const float *gsrc) {
    unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(sa), "l"(gsrc));
}
TTS_DEV void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

// Rank-one input mode: the scalar inputs x[b, t] of a CTA's R rows are staged in shared memory in windows
// of XW timesteps (cp.async, double-buffered) instead of being carried in registers one step ahead: the
// recurrent kernels run at the 255-register limit and the compiler was spilling those prefetch registers,
// which turned every prefetch into a synchronous wait on its own load (ncu: STL stalled on long scoreboard).
constexpr int XW = 32;
template <int R>
TTS_DEV void x1_fetch_window(float *__restrict__ dst, const float *__restrict__ x1, long long bstride, long long row0,
                             long long B, int steps, int w, int tid) {
    for (int e = tid; e < R * XW; e += NTHR) {
        const int b = e / XW, j = e % XW;
        const int tl = w * XW + j;
        if (row0 + b < B && tl < steps) cp_async4(dst + e, x1 + (row0 + b) * bstride + tl);
        else dst[e] = 0.f;
    }
}

// Packed FP32x2 FMA (Blackwell FFMA2): c.lo += a*w.lo, c.hi += a*w.hi with a scalar `a` operand.  Same FLOP
// rate as FFMA (measured 74.1 vs 72.5 TFLOP/s, tools/ffma2_probe.cu) for half the issue slots, which is what
// these LDS-fed register-tile loops are short of.
typedef unsigned long long f32x2;
TTS_DEV f32x2 pk2(float lo, float hi) {
    f32x2 v;
    asm("mov.b64 %0, {%1, %2};" : "=l"(v) : "f"(lo), "f"(hi));
    return v;
}
TTS_DEV void upk2(f32x2 v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
TTS_DEV void ffma2(f32x2 &c, float a, f32x2 w) {
    f32x2 aa;
    asm("mov.b64 %0, {%1, %1};" : "=l"(aa) : "f"(a));
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(c) : "l"(aa), "l"(w));
}

TTS_DEV float4 ld4(const float *p) { return *reinterpret_cast<const float4 *>(p); }
TTS_DEV void st4(float *p, float4 v) { *reinterpret_cast<float4 *>(p) = v; }

// ---------------------------------------------------------------------------------------------
// Shape: struct with static constexpr D, G, J[], I[], RK[] (ranks r_0..r_d)
// ---------------------------------------------------------------------------------------------
// floats per batch row of the X_k slot (i-block padded, see St::PAD); the runtime-indexed twin of St<S, k>::BS
template <class S>
constexpr int slot_floats_of(int k) {
    int m = 1;
    for (int q = k + 1; q < S::D; ++q) m *= S::I[q];
    for (int q = 0; q < k; ++q) m *= S::J[q];
    const int ks = cpad(cr4(S::J[k] * S::RK[k + 1]));
    const int nb = (k + 1 < S::D) ? S::I[k + 1] : 1;
    const int rb = m / nb;
    const int pad = (nb > 1 && ((rb * ks / 4) % 2 == 0)) ? 4 : 0;
    return nb * (rb * ks + pad);
}

template <class S, int k>
struct St {
    static_assert(k >= 0 && k < S::D, "stage index");
    static constexpr int J = S::J[k], I = S::I[k], r = S::RK[k], rn = S::RK[k + 1];
    static constexpr int Kraw = J * rn;               // contraction length in the blob
    static constexpr int K = cr4(Kraw);               // compute length (zero-padded; only a last stage with odd j needs it)
    static constexpr int N = I * r;
    static constexpr bool PACK = (S::G > 0);          // gate-interleaved layout of stage 0 (recurrent hh chains)
    static constexpr int mrow() {
        int m = 1;
        for (int q = k + 1; q < S::D; ++q) m *= S::I[q];
        for (int q = 0; q < k; ++q) m *= S::J[q];
        return m;
    }
    static constexpr int Mrow = mrow();
    static constexpr int KS = cpad(K);
    // The leading row index of X_k (k < d-1) is i_{k+1}: NB blocks of RB rows.  A stage writes X_k with lanes
    // running over i_{k+1} (and the core-gradient / data-gradient stages read it that way), so the block stride
    // must be an odd number of float4s or those accesses collapse onto one bank group (measured on the d3r8 chain:
    // 8-way conflicts, 33 % excess wavefronts in bwd_weight_stage).  PAD floats are inserted after every block.
    static constexpr int NB = (k + 1 < S::D) ? S::I[(k + 1 < S::D) ? k + 1 : 0] : 1;
    static constexpr int RB = Mrow / NB;
    static constexpr int PAD = (NB > 1 && ((RB * KS / 4) % 2 == 0)) ? 4 : 0;
    static constexpr int IBS = RB * KS + PAD;         // block stride
    static constexpr int BS = NB * IBS;               // floats per batch row of X_k
    TT_HD static constexpr int roff(int row) { return row * KS + (row / RB) * PAD; }   // offset of row `row`
    static_assert(BS == slot_floats_of<S>(k), "slot size formulas must agree");
    // shared-memory weight layout: k >= 1: [kappa][n] stride NS;  k == 0: [kappa][i0'][4 gates]
    static constexpr int NW = (k == 0 && PACK) ? (I / (PACK ? S::G : 1)) * 4 : N;
    static constexpr int NS = cpad(NW);
    static constexpr int WFLOATS = cr4(K * NS);
    static constexpr int CORE = r * I * J * rn;       // floats of core k in the blob
};

// Column of gate g of first-mode slice i0' in the gate-packed stage-0 layouts (W_0, W_0^T rows, dY_0):
//   LSTM (G = 4):            i0'*4 + g
//   GRU  (G = 3), I0' even:  slices are packed in pairs so that FFMA2 lanes carry no padding:
//                            [r0 z0 r1 z1 | n0 n1 - -] per pair of slices  ("pair packing")
//   GRU, I0' odd:            i0'*4 + g with the 4th column unused
template <class S> constexpr bool gru_pairs() { return S::G == 3 && ((S::I[0] / 3) % 2 == 0); }
template <class S> TT_HD constexpr int gate_col(int i0p, int g) {
    if (gru_pairs<S>()) {
        const int p = i0p / 2, e = i0p % 2;
        return (g < 2) ? p * 8 + e * 2 + g : p * 8 + 4 + e;
    }
    return i0p * 4 + g;
}
template <class S> TT_HD constexpr bool gate_col_valid(int col) {
    if (S::G == 4) return true;
    return gru_pairs<S>() ? (col % 8) < 6 : (col % 4) != 3;
}

template <class S> constexpr int n_in() { int v = 1; for (int k = 0; k < S::D; ++k) v *= S::J[k]; return v; }
template <class S> constexpr int n_out() { int v = 1; for (int k = 0; k < S::D; ++k) v *= S::I[k]; return v; }

template <class S, int k> struct WOff { static constexpr int v = WOff<S, k - 1>::v + St<S, k - 1>::WFLOATS; };
template <class S> struct WOff<S, 0> { static constexpr int v = 0; };
template <class S> constexpr int w_floats() { return WOff<S, S::D - 1>::v + St<S, S::D - 1>::WFLOATS; }
template <class S, int k> struct COff { static constexpr int v = COff<S, k - 1>::v + St<S, k - 1>::CORE; };
template <class S> struct COff<S, 0> { static constexpr int v = 0; };
template <class S> constexpr int core_floats() { return COff<S, S::D - 1>::v + St<S, S::D - 1>::CORE; }

// ---- contracted chain: cores 0 and 1 of a three-core shape merged into one core ------------------
//   W01[i0*I1 + i1][j0*J1 + j1][a2] = sum_a1 G0[i0][j0][a1] G1[a1][i1][j1][a2]
// Adjacent modes merge in row-major order, so h_t keeps its [J0*J1][J2] layout in the first stage and the gate
// stays the high part of the first output mode: the two-core chain over (W01, G2) computes the same W_hh h with
// one stage, one block barrier and one shared-memory round trip fewer per step (d3 r8: 589 824 instead of
// 655 360 FLOPs per row-step).  The kernels read the original three-core blob and contract while staging;
// parameter and gradient blobs keep the three-core layout.
template <class S3>
struct Merge01 {
    static_assert(S3::D == 3 && S3::RK[0] == 1 && S3::RK[3] == 1, "Merge01 contracts cores 0 and 1 of a three-core chain");
    using Src = S3;
    static constexpr int D = 2, G = S3::G;
    static constexpr int J[7] = {S3::J[0] * S3::J[1], S3::J[2]};
    static constexpr int I[7] = {S3::I[0] * S3::I[1], S3::I[2]};
    static constexpr int RK[7] = {1, S3::RK[2], 1};
};
// shape whose blob the kernels of S read (S itself, or the three-core source of a Merge01)
template <class S, class = void> struct SrcOf { using type = S; static constexpr bool merged = false; };
template <class S> struct SrcOf<S, std::void_t<typename S::Src>> { using type = typename S::Src; static constexpr bool merged = true; };
template <class S> constexpr int blob_floats() { return core_floats<typename SrcOf<S>::type>(); }

// element e (blob order r,i,j,r') of core k of S; a contracted core is summed over a1 in a fixed order, so every CTA
// and both directions stage bit-identical weights
template <class S, int k>
TTS_DEV float core_elem(const float *__restrict__ cores, int e) {
    if constexpr (SrcOf<S>::merged) {
        using S3 = typename SrcOf<S>::type;
        if constexpr (k == 0) {
            using T = St<S, 0>;
            constexpr int J1 = S3::J[1], I1 = S3::I[1], R1 = S3::RK[1], R2 = S3::RK[2];
            const int ap = e % T::rn;
            const int t = e / T::rn;
            const int j = t % T::J, i = t / T::J;              // r_0 = 1
            const float *g0 = cores + COff<S3, 0>::v + ((i / I1) * S3::J[0] + j / J1) * R1;
            const float *g1 = cores + COff<S3, 1>::v + ((i % I1) * J1 + j % J1) * R2 + ap;
            float s = 0.f;
#pragma unroll
            for (int a1 = 0; a1 < R1; ++a1) s = fmaf(__ldg(g0 + a1), __ldg(g1 + a1 * (I1 * J1 * R2)), s);
            return s;
        } else {
            return __ldg(cores + COff<S3, k + 1>::v + e);
        }
    } else {
        return __ldg(cores + COff<S, k>::v + e);
    }
}

// ---- stage the cores: blob (r,i,j,r') -> shared W layouts --------------------------------------
template <class S, int k>
TTS_DEV void stage_weights_k(const float *__restrict__ cores, float *__restrict__ wsm, int tid) {
    using T = St<S, k>;
    constexpr int I0p = T::PACK ? T::I / (T::PACK ? S::G : 1) : 1;
    if (T::K != T::Kraw)         // zero rows of a padded contraction
        for (int e = tid; e < (T::K - T::Kraw) * T::NS; e += NTHR) wsm[WOff<S, k>::v + T::Kraw * T::NS + e] = 0.f;
    if (k == 0 && S::G == 3) {   // padded gate columns are read as zeros
        for (int e = tid; e < T::WFLOATS; e += NTHR) wsm[WOff<S, 0>::v + e] = 0.f;
        __syncthreads();
    }
    for (int e = tid; e < T::CORE; e += NTHR) {
        const int ap = e % T::rn;
        int t = e / T::rn;
        const int j = t % T::J;
        t /= T::J;
        const int i = t % T::I;
        const int a = t / T::I;
        int col;
        if (k == 0 && T::PACK) col = gate_col<S>(i % I0p, i / I0p);   // gate index = i / I0p (gates are the high part of i_0)
        else col = i * T::r + a;
        wsm[WOff<S, k>::v + (j * T::rn + ap) * T::NS + col] = core_elem<S, k>(cores, e);
    }
    if constexpr (k + 1 < S::D) stage_weights_k<S, k + 1>(cores, wsm, tid);
}

// ---------------------------------------------------------------------------------------------
// Lane arrangement.  Measured on B200 (tools/lds_probe.cu): an LDS.128 costs 2 wavefronts when the
// lanes that share an address are adjacent pairs (address = f(lane/2)) or when the address
// depends only on lane%2 and on the high lane bits; period-4/8/16 interleaved duplicates cost 4.
// So a warp is laid out as LX "x" positions (lane bits 1..lgLX) times LY = 32/LX "y" positions
// (lane bit 0 and the top bits): the x operand is read pair-blocked, the y operand with period 2.
// ---------------------------------------------------------------------------------------------
template <int LX>
struct Lanes {
    static constexpr int LY = 32 / LX;
    static constexpr int lg = (LX == 32) ? 5 : (LX == 16) ? 4 : (LX == 8) ? 3 : (LX == 4) ? 2 : (LX == 2) ? 1 : 0;
    TTS_DEV static int x(int lane) { return (LX == 32) ? lane : ((lane >> 1) & (LX - 1)); }
    TTS_DEV static int y(int lane) { return (LX == 32) ? 0 : ((lane & 1) | ((lane >> (1 + lg)) << 1)); }
};

// ---------------------------------------------------------------------------------------------
// Forward stage k >= 1:  X_{k-1}[(i,m,a)] = sum_kappa X_k[m][kappa] W_k[kappa][(i,a)]
// thread tile = (R batch rows x TMr rows) x TN columns; TMr rows are MTl apart (lanes read
// neighbouring rows), the TN = 8 columns are two float4 groups N/2 apart (lanes read neighbouring
// float4s of W).  x = column tile, y = row tile.
// ---------------------------------------------------------------------------------------------
template <class S, int k, int R, int TMr_, int TN_>
struct FwdMap {
    using T = St<S, k>;
    static constexpr int TN = TN_, TMr = TMr_;
    static_assert(TN == 4 || TN == 8, "TN");
    static_assert(T::K % 4 == 0 && T::N % TN == 0 && T::r % 4 == 0, "static path needs K, N, r multiples of 4");
    static_assert(T::Mrow % TMr == 0, "TMr must divide Mrow");
    static constexpr int NTl = T::N / TN;
    static constexpr int MTl = T::Mrow / TMr;
    static constexpr int LX = p2div(NTl, 16);                  // column tiles across a warp: largest power of two <= 16 dividing NTl
    static constexpr int LY = 32 / LX;
    static_assert(NTl % LX == 0 && MTl % LY == 0, "tile grid must be a multiple of the lane grid");
    static constexpr int WX = NTl / LX;                         // warps along columns
    static constexpr int TT = MTl * NTl;
    static constexpr int ITER = (TT + NTHR - 1) / NTHR;
    static_assert(TT % NTHR == 0 || TT < NTHR, "tile count");
};

template <class S, int k, int R, int TMr, int TN>
TTS_DEV void fwd_stage(const float *__restrict__ X, const float *__restrict__ W, float *__restrict__ Y, int tid) {
    using T = St<S, k>;
    using To = St<S, k - 1>;
    using M = FwdMap<S, k, R, TMr, TN>;
    using L = Lanes<M::LX>;
    constexpr int Jp = To::J, KSo = To::KS, BSo = To::BS;
    constexpr int ISo = To::IBS;
    static_assert(To::RB == T::Mrow / Jp, "i-block rows of the output slot");
    // rows q*MTl + mt of X_k: separable offsets when whole blocks lie between consecutive q
    constexpr bool SEP = (T::PAD == 0) || (M::MTl % T::RB == 0);
    constexpr int QS = M::MTl * T::KS + (M::MTl / T::RB) * T::PAD;
    constexpr int NG = TN / 4;                 // float4 column groups per thread
    constexpr int GSTR = T::N / NG;            // distance between the groups (columns)
    const int lane = tid & 31, warp = tid >> 5;
#pragma unroll 1
    for (int it = 0; it < M::ITER; ++it) {
        const int wv = warp + it * (NTHR / 32);
        const int tn = (wv % M::WX) * M::LX + L::x(lane);
        const int mt = (wv / M::WX) * M::LY + L::y(lane);
        if (M::TT < NTHR && mt >= M::MTl) break;
        f32x2 acc2[R][TMr][TN / 2];
#pragma unroll
        for (int b = 0; b < R; ++b)
#pragma unroll
            for (int q = 0; q < TMr; ++q)
#pragma unroll
                for (int j = 0; j < TN / 2; ++j) acc2[b][q][j] = 0ull;
        const float *xb = X + T::roff(mt);
        const float *wb = W + tn * 4;
        int xq[TMr];
#pragma unroll
        for (int q = 0; q < TMr; ++q) xq[q] = SEP ? q * QS : T::roff(mt + q * M::MTl) - T::roff(mt);
#pragma unroll(unroll_of(T::K / 4))
        for (int k4 = 0; k4 < T::K; k4 += 4) {
            float4 a[R][TMr];
#pragma unroll
            for (int b = 0; b < R; ++b)
#pragma unroll
                for (int q = 0; q < TMr; ++q) a[b][q] = ld4(xb + b * T::BS + xq[q] + k4);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                f32x2 w2[TN / 2];
#pragma unroll
                for (int g = 0; g < NG; ++g) {
                    const float4 t = ld4(wb + (k4 + kk) * T::NS + g * GSTR);
                    w2[2 * g] = pk2(t.x, t.y);
                    w2[2 * g + 1] = pk2(t.z, t.w);
                }
#pragma unroll
                for (int b = 0; b < R; ++b)
#pragma unroll
                    for (int q = 0; q < TMr; ++q) {
                        const float av = kk == 0 ? a[b][q].x : (kk == 1 ? a[b][q].y : (kk == 2 ? a[b][q].z : a[b][q].w));
#pragma unroll
                        for (int j = 0; j < TN / 2; ++j) ffma2(acc2[b][q][j], av, w2[j]);
                    }
            }
        }
#pragma unroll
        for (int q = 0; q < TMr; ++q) {
            const int mr = q * M::MTl + mt;
            const int base = (mr / Jp) * KSo + (mr % Jp) * T::r;
#pragma unroll
            for (int g = 0; g < NG; ++g) {
                const int n = g * GSTR + tn * 4;
                const int off = base + (n / T::r) * ISo + (n % T::r);
#pragma unroll
                for (int b = 0; b < R; ++b) {
                    float4 v;
                    upk2(acc2[b][q][2 * g], v.x, v.y);
                    upk2(acc2[b][q][2 * g + 1], v.z, v.w);
                    st4(Y + b * BSo + off, v);
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Final stage (k = 0): every gate of a hidden unit ends up in one thread.
//   thread tile  = (R batch rows x TMr rows) x (TI first-mode slices x G gates), over 1/SK of K
//   thread grid  = MTl row tiles x ITl slice tiles x SK k-splits = NTHR threads
//   lanes        = 16 row tiles (x) x 2 slice tiles (y)   [ITl >= 2]   or 32 row tiles [ITl == 1]
//   after the k-loop the SK partial tiles are reduce-scattered through shared memory: thread kh
//   keeps the elements e = q*TI + i with e % SK == kh (NE = TMr*TI/SK of them).
// hidden unit of (mr, i0') is  h = i0' * Mrow_0 + mr
// ---------------------------------------------------------------------------------------------
template <class S, int R, int TMr_, int TI_, int SK_>
struct FinMap {
    using T = St<S, 0>;
    static_assert(T::r == 1 && T::I % S::G == 0, "gates must align with the first output mode");
    static_assert(!gru_pairs<S>() || TI_ % 2 == 0, "GRU pair packing needs an even number of slices per thread");
    static constexpr int TMr = TMr_, TI = TI_, SK = SK_;
    static constexpr int I0p = T::I / S::G;
    static_assert(I0p % TI == 0 && T::Mrow % TMr == 0 && (T::K / 4) % SK == 0, "final tile shape");
    static_assert((TMr * TI) % SK == 0, "k-split must divide the tile elements");
    static constexpr int ITl = I0p / TI;
    static constexpr int MTl = T::Mrow / TMr;
    static constexpr int TT = MTl * ITl * SK;
    static_assert(TT == NTHR, "final stage must use exactly one tile per thread");
    static constexpr int NE = TMr * TI / SK;            // elements (hidden units per batch row) owned per thread
    static constexpr int LX = (ITl >= 2) ? 16 : 32;
    static constexpr int LYI = (ITl >= 2) ? 2 : 1;      // slice tiles per warp
    static_assert(MTl % LX == 0 && ITl % LYI == 0, "lane grid");
    static constexpr int WM = MTl / LX;                 // warps along rows
    static constexpr int WI = ITl / LYI;                // warps along slices
    static constexpr int KPART = T::K / SK;
    static constexpr int XCH = (SK > 1) ? cr4((SK - 1) * NE * R * 4) : 0;   // exchange floats per thread
    static constexpr int XCH_FLOATS = XCH * NTHR;
    TTS_DEV static void coords(int tid, int &mt, int &itg, int &kh) {
        const int lane = tid & 31, warp = tid >> 5;
        using L = Lanes<LX>;
        mt = (warp % WM) * LX + L::x(lane);
        itg = ((warp / WM) % WI) * LYI + L::y(lane);
        kh = warp / (WM * WI);
    }
    // element e = q*TI + i  ->  hidden unit
    TTS_DEV static int hidden(int mt, int itg, int e) {
        const int q = e / TI, i = e % TI;
        return (itg * TI + i) * T::Mrow + q * MTl + mt;
    }
};

// accumulates the partial tile of this thread; acc[b][q][i][g]
template <class S, int R, class FM>
TTS_DEV void final_partial(const float *__restrict__ X, const float *__restrict__ W, int mt, int itg, int kh,
                           float (&acc)[R][FM::TMr][FM::TI][4]) {
    using T = St<S, 0>;
    constexpr int TMr = FM::TMr, TI = FM::TI;
    constexpr bool SEP = (T::PAD == 0) || (FM::MTl % T::RB == 0);
    constexpr int QS = FM::MTl * T::KS + (FM::MTl / T::RB) * T::PAD;
    const float *xb = X + T::roff(mt) + kh * FM::KPART;
    int xq[TMr];
#pragma unroll
    for (int q = 0; q < TMr; ++q) xq[q] = SEP ? q * QS : T::roff(mt + q * FM::MTl) - T::roff(mt);
    const float *wb = W + kh * FM::KPART * T::NS + itg * TI * 4;
    f32x2 acc2[R][TMr][TI][2];
#pragma unroll
    for (int b = 0; b < R; ++b)
#pragma unroll
        for (int q = 0; q < TMr; ++q)
#pragma unroll
            for (int i = 0; i < TI; ++i) { acc2[b][q][i][0] = 0ull; acc2[b][q][i][1] = 0ull; }
#pragma unroll(unroll_of(FM::KPART / 4))
    for (int k4 = 0; k4 < FM::KPART; k4 += 4) {
        float4 a[R][TMr];
#pragma unroll
        for (int b = 0; b < R; ++b)
#pragma unroll
            for (int q = 0; q < TMr; ++q) a[b][q] = ld4(xb + b * T::BS + xq[q] + k4);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            f32x2 w2[TI][2];
#pragma unroll
            for (int i = 0; i < TI; ++i) {
                const float4 t = ld4(wb + (k4 + kk) * T::NS + i * 4);
                w2[i][0] = pk2(t.x, t.y);
                w2[i][1] = pk2(t.z, t.w);          // GRU: (n gate, zero pad)
            }
#pragma unroll
            for (int b = 0; b < R; ++b)
#pragma unroll
                for (int q = 0; q < TMr; ++q) {
                    const float av = kk == 0 ? a[b][q].x : (kk == 1 ? a[b][q].y : (kk == 2 ? a[b][q].z : a[b][q].w));
#pragma unroll
                    for (int i = 0; i < TI; ++i) {
                        ffma2(acc2[b][q][i][0], av, w2[i][0]);
                        // GRU pair packing: the 4th pair of every slice pair is padding
                        if (!(gru_pairs<S>() && (i % 2 == 1))) ffma2(acc2[b][q][i][1], av, w2[i][1]);
                    }
                }
        }
    }
#pragma unroll
    for (int b = 0; b < R; ++b)
#pragma unroll
        for (int q = 0; q < TMr; ++q)
#pragma unroll
            for (int i = 0; i < TI; ++i) {
                if (gru_pairs<S>()) {
                    // columns of a slice pair: [r0 z0 | r1 z1 | n0 n1 | - -]; slice i reads pair (i%2) and half of pair 2
                    const int i0 = i & ~1;
                    float lo, hi;
                    upk2(acc2[b][q][i0][i % 2], acc[b][q][i][0], acc[b][q][i][1]);
                    upk2(acc2[b][q][i0 + 1][0], lo, hi);
                    acc[b][q][i][2] = (i % 2 == 0) ? lo : hi;
                    acc[b][q][i][3] = 0.f;
                } else {
                    upk2(acc2[b][q][i][0], acc[b][q][i][0], acc[b][q][i][1]);
                    upk2(acc2[b][q][i][1], acc[b][q][i][2], acc[b][q][i][3]);
                }
            }
}

// reduce-scatter of the SK partial tiles: on return pre[b][n][g] holds the full sums of the NE
// elements this thread owns (element index e = n*SK + kh).  xch: FM::XCH_FLOATS floats of shared
// memory; contains two block barriers when SK > 1.
template <class S, int R, class FM>
TTS_DEV void final_reduce(float (&acc)[R][FM::TMr][FM::TI][4], float (&pre)[R][FM::NE][4], float *xch, int tid, int kh) {
    constexpr int TI = FM::TI, SK = FM::SK, NE = FM::NE;
    constexpr int PER = NTHR / SK;                       // threads per k-split group
    if constexpr (SK > 1) {
        // slot layout: [(d-1)][n][b] float4 per thread, thread-minor: xch4[slot * NTHR + owner_tid]
        float4 *x4 = reinterpret_cast<float4 *>(xch);
        const int tprime = tid % PER;
#pragma unroll
        for (int e = 0; e < FM::TMr * TI; ++e) {
            const int owner = e % SK;                    // compile-time after unrolling
            const int n = e / SK;
            const int q = e / TI, i = e % TI;
            // this thread is the dlt-th partner of `owner`, dlt = (kh - owner) mod SK (warp-uniform; 0 = it owns e):
            // one uniform branch per element, the slot index only enters the address
            const int dlt = (kh - owner + SK) % SK;
            if (dlt != 0) {
                float4 *dst = x4 + ((dlt - 1) * NE * R + n * R) * NTHR + owner * PER + tprime;
#pragma unroll
                for (int b = 0; b < R; ++b)
                    dst[b * NTHR] = make_float4(acc[b][q][i][0], acc[b][q][i][1], acc[b][q][i][2], acc[b][q][i][3]);
            }
        }
        __syncthreads();
#pragma unroll
        for (int e = 0; e < FM::TMr * TI; ++e) {
            const int owner = e % SK;
            const int n = e / SK;
            const int q = e / TI, i = e % TI;
            if (owner == kh) {
#pragma unroll
                for (int b = 0; b < R; ++b) {
                    float s0 = acc[b][q][i][0], s1 = acc[b][q][i][1], s2 = acc[b][q][i][2], s3 = acc[b][q][i][3];
#pragma unroll
                    for (int dlt = 1; dlt < SK; ++dlt) {
                        const float4 v = x4[((dlt - 1) * NE * R + n * R + b) * NTHR + tid];
                        s0 += v.x; s1 += v.y; s2 += v.z; s3 += v.w;
                    }
                    pre[b][n][0] = s0; pre[b][n][1] = s1; pre[b][n][2] = s2; pre[b][n][3] = s3;
                }
            }
        }
    } else {
#pragma unroll
        for (int e = 0; e < FM::TMr * TI; ++e) {
            const int q = e / TI, i = e % TI;
#pragma unroll
            for (int b = 0; b < R; ++b)
#pragma unroll
                for (int g = 0; g < 4; ++g) pre[b][e][g] = acc[b][q][i][g];
        }
    }
}

#ifndef TTS_ACCURATE_GATES
// MUFU-based logistic (ex2.approx + rcp.approx): measured parity error stays at 1-4e-7 forward and
// <= 7e-7 on gradients (tools/parity_report.py), bars are 1e-5 / 1e-4.  -DTTS_ACCURATE_GATES restores expf + IEEE division.
TTS_DEV float sigmoidf_acc(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
// branch-free tanh: odd minimax polynomial on |x| < 0.6 (max rel err 8e-8), 1 - 2/(e^{2|x|}+1) beyond
// (libdevice tanhf takes the same two routes but branches, which diverges inside a warp)
TTS_DEV float tanh_g(float x) {
    const float ax = fabsf(x);
    const float p = x * x;
    float r = fmaf(p, -0.00598506f, 0.02086822f);
    r = fmaf(r, p, -0.05380359f);
    r = fmaf(r, p, 0.13332133f);
    r = fmaf(r, p, -0.33333305f);
    const float small = fmaf(x * p, r, x);
    const float e = __expf(2.0f * ax);
    const float big = copysignf(1.0f - __fdividef(2.0f, e + 1.0f), x);
    return ax < 0.6f ? small : big;
}
#else
TTS_DEV float sigmoidf_acc(float x) { return 1.0f / (1.0f + expf(-x)); }
TTS_DEV float tanh_g(float x) { return tanhf(x); }
#endif

// ---- per (shape, R) tuning table ----------------------------------------------------------------
// TMr[k], TN[k] for the forward stages k >= 1; FTMr / FTI / FSK for the final stage
template <int FTMr_, int FTI_, int FSK_, int TM1 = 1, int TN1 = 8, int TM2 = 1, int TN2 = 8, int TM3 = 1, int TN3 = 8>
struct Tune {
    static constexpr int FTMr = FTMr_, FTI = FTI_, FSK = FSK_;
    static constexpr int TMr[4] = {0, TM1, TM2, TM3};
    static constexpr int TN[4] = {0, TN1, TN2, TN3};
};

// ping-pong slots of a forward-only chain: P holds X_{d-2}, X_{d-4}, ..; Q holds X_{d-3}, ..
template <class S, int R>
struct PPSlots {
    static constexpr int D = S::D;
    static constexpr int pfloats() {
        int m = 0;
        if (D >= 2) m = cmax(m, St<S, (D >= 2 ? D - 2 : 0)>::BS);
        if (D >= 4) m = cmax(m, St<S, (D >= 4 ? D - 4 : 0)>::BS);
        if (D >= 6) m = cmax(m, St<S, (D >= 6 ? D - 6 : 0)>::BS);
        return cr4(R * m);
    }
    static constexpr int qfloats() {
        int m = 0;
        if (D >= 3) m = cmax(m, St<S, (D >= 3 ? D - 3 : 0)>::BS);
        if (D >= 5) m = cmax(m, St<S, (D >= 5 ? D - 5 : 0)>::BS);
        return cr4(R * m);
    }
    static constexpr int P = pfloats(), Q = qfloats();
};

// shared-memory floats of the forward recurrent kernel
template <class S, int R, class TU>
struct FwdSmem {
    static constexpr int D = S::D;
    using FM = FinMap<S, R, TU::FTMr, TU::FTI, TU::FSK>;
    static constexpr int W = w_floats<S>();
    static constexpr int HS = cr4(R * St<S, D - 1>::BS);
    static constexpr int pfloats() {
        int m = 0;
        if (D >= 2) m = cmax(m, St<S, (D >= 2 ? D - 2 : 0)>::BS);
        if (D >= 4) m = cmax(m, St<S, (D >= 4 ? D - 4 : 0)>::BS);
        if (D >= 6) m = cmax(m, St<S, (D >= 6 ? D - 6 : 0)>::BS);
        return cr4(R * m);
    }
    static constexpr int qfloats() {
        int m = 0;
        if (D >= 3) m = cmax(m, St<S, (D >= 3 ? D - 3 : 0)>::BS);
        if (D >= 5) m = cmax(m, St<S, (D >= 5 ? D - 5 : 0)>::BS);
        return cr4(R * m);
    }
    static constexpr int P = pfloats(), Q = qfloats();
    static constexpr int XCH = FM::XCH_FLOATS;
    static constexpr int X1W = 2 * R * XW;               // rank-one input windows
    static constexpr int TOTAL = W + HS + P + Q + XCH + X1W;
    static constexpr size_t BYTES = (size_t)TOTAL * 4;
};

struct RnnFwdSArgs {
    int steps;
    long long B;
    const float *xg;         // (B, steps, G*H) ih projection (+ biases folded for LSTM); MODE_XG
    long long xg_bstride;
    const float *x1;         // rank-one input mode: x (B, T, 1) pre-offset to this chunk; row stride x1_bstride
    long long x1_bstride;
    const float *w_eff;      // rank-one input mode: (G*H) dense column of W_ih
    const float *bias_ih;    // rank-one mode: (G*H) or null
    const float *cores;      // hh core blob
    const float *bias_hh;    // (G*H) or null: GRU always; LSTM only in rank-one mode (else folded into xg)
    const float *h_in, *c_in;
    float *out;
    long long out_bstride;
    float *c_save;
    float *h_out, *c_out;
    // optional (training): keep the gate activations of every step so that backward skips the final stage of the
    // chain recompute.  Row b, step t at  base + b*bstride + t*per_step.
    float *u_save;           // per step: H x 4 floats [h][gate]: the gate activations (LSTM i,f,g,o; GRU r,z,n and u_n)
    long long u_bstride;
};

enum { MODE_XG = 0, MODE_RANK1 = 1 };

// run stages D-1 .. 1 (each followed by a barrier); returns the slot holding X_0
template <class S, int R, class TU, int k>
TTS_DEV const float *fwd_chain_pp(float *hs, float *P, float *Q, const float *wsm, int tid) {
    if constexpr (k == 0) {
        return (S::D == 1) ? hs : (((S::D - 2) % 2 == 0) ? P : Q);
    } else {
        const float *X = (k == S::D - 1) ? hs : (((S::D - 2 - k) % 2 == 0) ? P : Q);
        float *Y = ((S::D - 2 - (k - 1)) % 2 == 0) ? P : Q;
        fwd_stage<S, k, R, TU::TMr[k], TU::TN[k]>(X, wsm + WOff<S, k>::v, Y, tid);
        __syncthreads();
        return fwd_chain_pp<S, R, TU, k - 1>(hs, P, Q, wsm, tid);
    }
}

template <class S, int CELL, int R, int MODE, class TU, int MINB = 1>
__global__ void __launch_bounds__(NTHR, MINB) k_rnn_fwd_s(const __grid_constant__ RnnFwdSArgs a) {
    extern __shared__ __align__(16) float smem[];
    using SM = FwdSmem<S, R, TU>;
    using FM = typename SM::FM;
    using TL = St<S, S::D - 1>;
    constexpr int G = S::G, H = n_in<S>(), GH = G * H;
    constexpr int NE = FM::NE;
    constexpr bool LSTM = (CELL == TTRNN_CELL_LSTM);
    static_assert(G == (LSTM ? 4 : 3), "gate count");
    const int tid = threadIdx.x;
    float *wsm = smem;
    float *hs = wsm + SM::W;
    float *P = hs + SM::HS;
    float *Q = P + SM::P;
    float *xch = Q + SM::Q;
    float *xw1 = xch + SM::XCH;

    stage_weights_k<S, 0>(a.cores, wsm, tid);

    int mt, itg, kh;
    FM::coords(tid, mt, itg, kh);
    // hidden units owned by this thread: element e = n*SK + kh
    int hid[NE];
    float bhh[NE][4], weff[NE][4], bih[NE][4];
#pragma unroll
    for (int n = 0; n < NE; ++n) {
        hid[n] = FM::hidden(mt, itg, n * FM::SK + kh);
#pragma unroll
        for (int g = 0; g < G; ++g) {
            const int col = g * H + hid[n];
            bhh[n][g] = a.bias_hh ? __ldg(a.bias_hh + col) : 0.f;
            weff[n][g] = (MODE == MODE_RANK1) ? __ldg(a.w_eff + col) : 0.f;
            bih[n][g] = (MODE == MODE_RANK1 && a.bias_ih) ? __ldg(a.bias_ih + col) : 0.f;
        }
    }

    const long long ntiles = (a.B + R - 1) / R;
    for (long long tile_i = blockIdx.x; tile_i < ntiles; tile_i += gridDim.x) {
        const long long row0 = tile_i * R;
        __syncthreads();
        // initial state: h -> shared slot (X_{d-1} layout), c / h_prev -> registers of the owner thread
        for (int e = tid; e < R * H; e += NTHR) {
            const int b = e / H, h = e % H;
            float hv = 0.f;
            if (row0 + b < a.B && a.h_in) hv = __ldg(a.h_in + (row0 + b) * H + h);
            hs[b * TL::BS + (h / TL::K) * TL::KS + (h % TL::K)] = hv;
        }
        float cst[R][NE], hpr[R][NE];
#pragma unroll
        for (int b = 0; b < R; ++b)
#pragma unroll
            for (int n = 0; n < NE; ++n) {
                const bool ok = (row0 + b < a.B);
                cst[b][n] = (LSTM && ok && a.c_in) ? __ldg(a.c_in + (row0 + b) * H + hid[n]) : 0.f;
                hpr[b][n] = (ok && a.h_in) ? __ldg(a.h_in + (row0 + b) * H + hid[n]) : 0.f;
            }
        if (MODE == MODE_RANK1) {
            x1_fetch_window<R>(xw1, a.x1, a.x1_bstride, row0, a.B, a.steps, 0, tid);
            cp_async_wait_all();
        }
        __syncthreads();
        // per-unit output pointers of this tile (advanced by one step at the end of every step) and the number
        // of valid rows: the per-step stores are then single predicated instructions with no 64-bit index
        // arithmetic and no branches between the gate computations of different rows
        const int nvalid = (a.B - row0 < R) ? (int)(a.B - row0) : R;
        float *out_p[NE], *cs_p[NE], *us_p[NE];
#pragma unroll
        for (int n = 0; n < NE; ++n) {
            out_p[n] = a.out + row0 * a.out_bstride + hid[n];
            cs_p[n] = (LSTM && a.c_save) ? a.c_save + row0 * a.out_bstride + hid[n] : nullptr;
            us_p[n] = a.u_save ? a.u_save + row0 * a.u_bstride + 4 * hid[n] : nullptr;
        }
        const bool have_cs = LSTM && a.c_save != nullptr, have_us = a.u_save != nullptr;

        // operands of the gate phase are fetched one step ahead (the loads of step t+1 are issued at the top
        // of step t and land while the chain of step t runs); rank-one inputs come from the shared windows
        float xin_n[R][NE][4];
        auto fetch_in = [&](int tl) {
            if (MODE == MODE_XG) {
#pragma unroll
                for (int b = 0; b < R; ++b)
#pragma unroll
                    for (int n = 0; n < NE; ++n)
#pragma unroll
                        for (int g = 0; g < G; ++g)
                            xin_n[b][n][g] = (b < nvalid)
                                ? __ldg(a.xg + row0 * a.xg_bstride + hid[n] + (long long)tl * GH + b * a.xg_bstride + g * H) : 0.f;
            }
        };
        fetch_in(0);
        for (int t = 0; t < a.steps; ++t) {
            float xin[R][NE][4];
            float x1[R];
#pragma unroll
            for (int b = 0; b < R; ++b) {
                x1[b] = (MODE == MODE_RANK1) ? xw1[((t / XW) & 1) * R * XW + b * XW + (t % XW)] : 0.f;
#pragma unroll
                for (int n = 0; n < NE; ++n)
#pragma unroll
                    for (int g = 0; g < 4; ++g) xin[b][n][g] = xin_n[b][n][g];
            }
            if (MODE == MODE_RANK1 && (t % XW) == 0 && t + XW < a.steps)
                x1_fetch_window<R>(xw1 + (((t / XW) + 1) & 1) * R * XW, a.x1, a.x1_bstride, row0, a.B, a.steps, t / XW + 1, tid);
            if (t + 1 < a.steps) fetch_in(t + 1);
            // ---- stages d-1 .. 1
            const float *X0 = fwd_chain_pp<S, R, TU, S::D - 1>(hs, P, Q, wsm, tid);
            // ---- stage 0 (split over K) + reduce-scatter + gate math + state update
            float pre[R][NE][4];
            {
                float acc[R][FM::TMr][FM::TI][4];
                final_partial<S, R, FM>(X0, wsm + WOff<S, 0>::v, mt, itg, kh, acc);
                final_reduce<S, R, FM>(acc, pre, xch, tid, kh);
            }
#pragma unroll
            for (int b = 0; b < R; ++b)
#pragma unroll
                for (int n = 0; n < NE; ++n) {
                    const int h = hid[n];
                    float ain[4];
#pragma unroll
                    for (int g = 0; g < G; ++g)
                        ain[g] = (MODE == MODE_XG) ? xin[b][n][g] : fmaf(x1[b], weff[n][g], bih[n][g]);
                    float keep[4];                      // gate activations kept for backward
                    float hnew;
                    if (LSTM) {
                        const float ig = sigmoidf_acc(pre[b][n][0] + bhh[n][0] + ain[0]);
                        const float fg = sigmoidf_acc(pre[b][n][1] + bhh[n][1] + ain[1]);
                        const float gg = tanh_g(pre[b][n][2] + bhh[n][2] + ain[2]);
                        const float og = sigmoidf_acc(pre[b][n][3] + bhh[n][3] + ain[3]);
                        const float cn = fg * cst[b][n] + ig * gg;
                        cst[b][n] = cn;
                        hnew = og * tanh_g(cn);
                        keep[0] = ig; keep[1] = fg; keep[2] = gg; keep[3] = og;
                    } else {
                        const float un = pre[b][n][2] + bhh[n][2];
                        const float rg = sigmoidf_acc(ain[0] + (pre[b][n][0] + bhh[n][0]));
                        const float zg = sigmoidf_acc(ain[1] + (pre[b][n][1] + bhh[n][1]));
                        const float ng = tanh_g(ain[2] + rg * un);
                        hnew = (1.0f - zg) * ng + zg * hpr[b][n];
                        keep[0] = rg; keep[1] = zg; keep[2] = ng; keep[3] = un;
                    }
                    const bool okb = b < nvalid;
                    if (okb && have_us)                  // [row][t][h][4]: one 16-byte store per hidden unit
                        st4(us_p[n] + b * a.u_bstride, make_float4(keep[0], keep[1], keep[2], keep[3]));
                    hpr[b][n] = hnew;
                    hs[b * TL::BS + (h / TL::K) * TL::KS + (h % TL::K)] = hnew;
                    if (okb) out_p[n][b * a.out_bstride] = hnew;
                    if (okb && have_cs) cs_p[n][b * a.out_bstride] = cst[b][n];
                }
#pragma unroll
            for (int n = 0; n < NE; ++n) {
                out_p[n] += H;
                if (have_cs) cs_p[n] += H;
                if (have_us) us_p[n] += 4 * H;
            }
            if (MODE == MODE_RANK1) cp_async_wait_all();
            __syncthreads();
        }
#pragma unroll
        for (int b = 0; b < R; ++b)
#pragma unroll
            for (int n = 0; n < NE; ++n)
                if (row0 + b < a.B) {
                    if (a.h_out) a.h_out[(row0 + b) * H + hid[n]] = hpr[b][n];
                    if (LSTM && a.c_out) a.c_out[(row0 + b) * H + hid[n]] = cst[b][n];
                }
    }
}

// =============================================================================================
// Backward (BPTT) -- static path
// =============================================================================================

// ---- transposed weights  WT_k[n][kappa]  (row stride cpad(K)); k == 0 rows are n = i0'*4 + gate ----
template <class S, int k>
struct StT {
    using T = St<S, k>;
    static constexpr int ROWS = T::NW;                 // n (k >= 1) or i0'*4+g (k == 0)
    static constexpr int KST = cpad(T::K);
    static constexpr int FLOATS = cr4(ROWS * KST);
};
template <class S, int k> struct WTOff { static constexpr int v = WTOff<S, k - 1>::v + StT<S, k - 1>::FLOATS; };
template <class S> struct WTOff<S, 0> { static constexpr int v = 0; };
template <class S> constexpr int wt_floats() { return WTOff<S, S::D - 1>::v + StT<S, S::D - 1>::FLOATS; }

template <class S, int k>
TTS_DEV void stage_weights_t(const float *__restrict__ cores, float *__restrict__ wt, int tid) {
    using T = St<S, k>;
    using TT_ = StT<S, k>;
    constexpr int I0p = T::PACK ? T::I / (T::PACK ? S::G : 1) : 1;
    constexpr bool ZERO = (k == 0 && S::G == 3) || (T::K != T::Kraw);
    if (ZERO)
        for (int e = tid; e < TT_::FLOATS; e += NTHR) wt[WTOff<S, k>::v + e] = 0.f;
    if (ZERO) __syncthreads();
    for (int e = tid; e < T::CORE; e += NTHR) {
        const int ap = e % T::rn;
        int t = e / T::rn;
        const int j = t % T::J;
        t /= T::J;
        const int i = t % T::I;
        const int a = t / T::I;
        const int row = (k == 0 && T::PACK) ? gate_col<S>(i % I0p, i / I0p) : i * T::r + a;
        wt[WTOff<S, k>::v + row * TT_::KST + j * T::rn + ap] = core_elem<S, k>(cores, e);
    }
    if constexpr (k + 1 < S::D) stage_weights_t<S, k + 1>(cores, wt, tid);
}

// ---------------------------------------------------------------------------------------------
// Backward-data stage:  dX_k[m][kappa] = sum_n dY_k[m][n] WT_k[n][kappa]
// Same register-tile structure as fwd_stage (rows x 8 columns, columns = kappa in two float4 groups
// K/2 apart, or one group when K < 8); the reduction runs over n in groups of four.
// SPLIT > 1 divides the reduction between SPLIT groups of warps; the partial tiles are
// reduce-scattered through shared memory (owner s keeps columns [s*CW, (s+1)*CW) of the tile).
//   k >= 1 : dY_k sits in the X_{k-1}-shaped buffer the forward stage wrote to
//   k == 0 : dY_0 is the gate-gradient buffer [b][mr][i0'*4+g], row stride DS0
// ---------------------------------------------------------------------------------------------
template <class S> struct DY0 {
    using T = St<S, 0>;
    static constexpr int DS = T::PACK ? cpad(T::NW) : T::NW; // row stride (plain chains: unpadded, saves shared memory)
    static constexpr int BS = T::Mrow * DS;                  // per batch row
};

template <class S, int k, int R, int TMr_, int SPLIT_>
struct BdMap {
    using T = St<S, k>;
    static constexpr int TMr = TMr_, SPLIT = SPLIT_;
    static constexpr int TN = (T::K % 8 == 0) ? 8 : 4;         // kappa columns per thread
    static constexpr int NG = TN / 4;
    static constexpr int GSTR = T::K / NG;
    static constexpr int CTl = T::K / TN;
    static constexpr int MTl = T::Mrow / TMr;
    static constexpr int RED = T::NW;                           // reduction length (incl. the padded gate of stage 0)
    static_assert(T::Mrow % TMr == 0 && (RED / 4) % SPLIT == 0, "bwd-data tile shape");
    static constexpr int LX = p2div(CTl, 16);                   // 12 column tiles (K = 96, H = 768 chains) -> 4 x 8 lanes
    static constexpr int LY = 32 / LX;
    static_assert(CTl % LX == 0 && MTl % LY == 0, "bwd-data lane grid");
    static constexpr int WX = CTl / LX;
    static constexpr int TT = MTl * CTl;                        // tiles per split
    static constexpr int PER = NTHR / SPLIT;                    // threads per split
    static constexpr int ITER = (TT + PER - 1) / PER;
    static_assert(TT % PER == 0 || TT < PER, "bwd-data tile count");
    static_assert(SPLIT == 1 || TT <= PER, "split stages use one tile per thread");
    static_assert(!(k == 0 && T::PACK) || SPLIT == 1 || S::G == 4, "stage 0 of a GRU chain must not be split");
    static constexpr int CW = TN / SPLIT > 0 ? TN / SPLIT : 1;  // columns kept per thread after the reduce-scatter
    static_assert(SPLIT == 1 || TN % SPLIT == 0, "split must divide the tile columns");
    static constexpr int XCH_FLOATS = (SPLIT > 1) ? (SPLIT - 1) * R * TMr * CW * NTHR : 0;
    static constexpr int REDP = RED / SPLIT;
};

template <class S, int k, int R, int TMr, int SPLIT>
TTS_DEV void bwd_data_stage(const float *__restrict__ dY, const float *__restrict__ WT, float *__restrict__ dX,
                            float *__restrict__ xch, int tid) {
    using T = St<S, k>;
    using M = BdMap<S, k, R, TMr, SPLIT>;
    using L = Lanes<M::LX>;
    constexpr int TN = M::TN, NG = M::NG, GSTR = M::GSTR;
    constexpr int KST = StT<S, k>::KST;
    // geometry of the dY buffer
    constexpr int Jp = (k == 0) ? 1 : St<S, (k == 0 ? 0 : k - 1)>::J;
    constexpr int KSo = (k == 0) ? DY0<S>::DS : St<S, (k == 0 ? 0 : k - 1)>::KS;
    constexpr int BSo = (k == 0) ? DY0<S>::BS : St<S, (k == 0 ? 0 : k - 1)>::BS;
    constexpr int ISo = (k == 0) ? 0 : St<S, (k == 0 ? 0 : k - 1)>::IBS;
    const int lane = tid & 31;
    const int sp = tid / M::PER;                 // split index (whole warps)
    const int wloc = (tid % M::PER) >> 5;
#pragma unroll 1
    for (int it = 0; it < M::ITER; ++it) {
        const int wv = wloc + it * (M::PER / 32);
        const int tn = (wv % M::WX) * M::LX + L::x(lane);
        const int mt = (wv / M::WX) * M::LY + L::y(lane);
        const bool live = !(M::TT < M::PER && mt >= M::MTl);
        float acc[R][TMr][TN];
        f32x2 acc2[R][TMr][TN / 2];
#pragma unroll
        for (int b = 0; b < R; ++b)
#pragma unroll
            for (int q = 0; q < TMr; ++q)
#pragma unroll
                for (int j = 0; j < TN / 2; ++j) acc2[b][q][j] = 0ull;
        if (live) {
            int rbase[TMr];
#pragma unroll
            for (int q = 0; q < TMr; ++q) {
                const int mr = q * M::MTl + mt;
                rbase[q] = (k == 0) ? mr * KSo : (mr / Jp) * KSo + (mr % Jp) * T::r;
            }
            const float *wb = WT + tn * 4;
            static_assert(k == 0 || M::REDP % T::r == 0 || T::r % M::REDP == 0 || SPLIT == 1, "split must align with the rank runs");
            const int nsp = sp * M::REDP;                             // first reduction index of this split
            const int abase = (k == 0) ? nsp : (nsp / T::r) * ISo + (nsp % T::r);
            const float *wsp = wb + nsp * KST;
#pragma unroll(unroll_of(M::REDP / 4))
            for (int n4 = 0; n4 < M::REDP; n4 += 4) {
                // nsp is a multiple of r (or the whole split lies inside one run), so the offset separates
                const int aoff = abase + ((k == 0) ? n4 : (n4 / T::r) * ISo + (n4 % T::r));
                const int n = n4;
                float4 a[R][TMr];
#pragma unroll
                for (int b = 0; b < R; ++b)
#pragma unroll
                    for (int q = 0; q < TMr; ++q) a[b][q] = ld4(dY + b * BSo + rbase[q] + aoff);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    if (k == 0 && T::PACK && !gate_col_valid<S>(n4 + kk)) continue;    // padded gate column (k = 0 is never split)
                    f32x2 w2[TN / 2];
#pragma unroll
                    for (int g = 0; g < NG; ++g) {
                        const float4 t = ld4(wsp + (n + kk) * KST + g * GSTR);
                        w2[2 * g] = pk2(t.x, t.y);
                        w2[2 * g + 1] = pk2(t.z, t.w);
                    }
#pragma unroll
                    for (int b = 0; b < R; ++b)
#pragma unroll
                        for (int q = 0; q < TMr; ++q) {
                            const float av = kk == 0 ? a[b][q].x : (kk == 1 ? a[b][q].y : (kk == 2 ? a[b][q].z : a[b][q].w));
#pragma unroll
                            for (int j = 0; j < TN / 2; ++j) ffma2(acc2[b][q][j], av, w2[j]);
                        }
                }
            }
        }
#pragma unroll
        for (int b = 0; b < R; ++b)
#pragma unroll
            for (int q = 0; q < TMr; ++q)
#pragma unroll
                for (int j = 0; j < TN / 2; ++j) upk2(acc2[b][q][j], acc[b][q][2 * j], acc[b][q][2 * j + 1]);
        if constexpr (SPLIT == 1) {
            if (live) {
#pragma unroll
                for (int q = 0; q < TMr; ++q) {
                    const int mr = q * M::MTl + mt;
#pragma unroll
                    for (int g = 0; g < NG; ++g)
#pragma unroll
                        for (int b = 0; b < R; ++b)
                            st4(dX + b * T::BS + T::roff(mr) + g * GSTR + tn * 4,
                                make_float4(acc[b][q][4 * g], acc[b][q][4 * g + 1], acc[b][q][4 * g + 2], acc[b][q][4 * g + 3]));
                }
            }
        } else {
            // reduce-scatter over the SPLIT groups: owner s keeps columns j in [s*CW, (s+1)*CW)
            constexpr int CW = M::CW;
            const int tprime = tid % M::PER;
#pragma unroll
            for (int j = 0; j < TN; ++j) {
                const int owner = j / CW, c = j % CW;
                // dlt = (sp - owner) mod SPLIT is warp-uniform (a split is a whole number of warps); 0 = own column.
                // One uniform branch per column; the partner index only enters the address.
                const int dlt = (sp - owner + SPLIT) % SPLIT;
                if (dlt != 0) {
                    float *dst = xch + (dlt - 1) * (R * TMr * CW * NTHR) + c * NTHR + owner * M::PER + tprime;
#pragma unroll
                    for (int b = 0; b < R; ++b)
#pragma unroll
                        for (int q = 0; q < TMr; ++q) dst[(b * TMr + q) * CW * NTHR] = acc[b][q][j];
                }
            }
            __syncthreads();
            if (live) {
#pragma unroll
                for (int j = 0; j < TN; ++j) {
                    const int owner = j / CW, c = j % CW;
                    if (owner == sp) {
                        const int col = (j / 4) * GSTR + tn * 4 + (j % 4);
#pragma unroll
                        for (int b = 0; b < R; ++b)
#pragma unroll
                            for (int q = 0; q < TMr; ++q) {
                                float sum = acc[b][q][j];
#pragma unroll
                                for (int dlt = 1; dlt < SPLIT; ++dlt)
                                    sum += xch[(((dlt - 1) * R + b) * TMr + q) * CW * NTHR + c * NTHR + tid];
                                dX[b * T::BS + T::roff(q * M::MTl + mt) + col] = sum;
                            }
                    }
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Backward-weight stage:  dW_k[kappa][n] += sum_m X_k[m][kappa] dY_k[m][n]
// Thread = (kappa tile of TK=8 | 4, n tile of 4, row group mg of MG); rows m = it*MG + mg.
// The TK x 4 tile stays in registers for the whole launch (no per-step reduction); the MG row
// groups are summed once at the end of the launch (flush_dw).
//   k == 0: n tile = the 4 (3 used) gates of one i0'
// ---------------------------------------------------------------------------------------------
template <class S, int k, int R, int TK_>
struct BwMap {
    using T = St<S, k>;
    static constexpr int TK = TK_;
    static_assert(TK == 4 || TK == 8, "TK");
    static constexpr int KT = T::K / TK;
    static constexpr int NT4 = T::NW / 4;                                 // n tiles (stage 0 of a gate chain: one i0')
    static constexpr int TILES = KT * NT4;
    static_assert(TILES <= NTHR && NTHR % TILES == 0, "bwd-weight tiles must divide the thread count");
    static constexpr int MG = NTHR / TILES;
    static constexpr int M = R * T::Mrow;
    static constexpr int ROWS = (M + MG - 1) / MG;                        // row iterations per thread
    // lanes: x = n tile (dY operand, pair-blocked), y = (kappa tile, row group) (X operand, period 2)
    static constexpr int LX = p2div(NT4, 16);
    static constexpr int LY = 32 / LX;
    static_assert(NT4 % LX == 0 && (KT * MG) % LY == 0, "bwd-weight lane grid");
    static constexpr int WXN = NT4 / LX;
    TTS_DEV static void coords(int tid, int &nt, int &kt, int &mg) {
        using L = Lanes<LX>;
        const int lane = tid & 31, warp = tid >> 5;
        nt = (warp % WXN) * LX + L::x(lane);
        const int rest = (warp / WXN) * LY + L::y(lane);
        kt = rest % KT;
        mg = rest / KT;
    }
};

template <class S, int k, int R, int TK>
TTS_DEV void bwd_weight_stage(const float *__restrict__ X, const float *__restrict__ dY, f32x2 (&acc2)[TK][2], int tid) {
    using T = St<S, k>;
    using M = BwMap<S, k, R, TK>;
    constexpr int Jp = (k == 0) ? 1 : St<S, (k == 0 ? 0 : k - 1)>::J;
    constexpr int KSo = (k == 0) ? DY0<S>::DS : St<S, (k == 0 ? 0 : k - 1)>::KS;
    constexpr int BSo = (k == 0) ? DY0<S>::BS : St<S, (k == 0 ? 0 : k - 1)>::BS;
    constexpr int ISo = (k == 0) ? 0 : St<S, (k == 0 ? 0 : k - 1)>::IBS;
    int nt, kt, mg;
    M::coords(tid, nt, kt, mg);
    const int n0 = nt * 4;
    const int yoff = (k == 0) ? n0 : (n0 / T::r) * ISo + (n0 % T::r);
    auto row_fma = [&](const float *xp, const float *yp) {
        const float4 y = ld4(yp);
        const f32x2 y01 = pk2(y.x, y.y), y23 = pk2(y.z, y.w);
        float x[TK];
#pragma unroll
        for (int g = 0; g < TK / 4; ++g) {
            const float4 t = ld4(xp + 4 * g);
            x[4 * g] = t.x; x[4 * g + 1] = t.y; x[4 * g + 2] = t.z; x[4 * g + 3] = t.w;
        }
#pragma unroll
        for (int a = 0; a < TK; ++a) {
            ffma2(acc2[a][0], x[a], y01);
            ffma2(acc2[a][1], x[a], y23);
        }
    };
    if constexpr (T::Mrow % M::MG == 0 && (k == 0 || M::MG % Jp == 0 || Jp % M::MG == 0) &&
                  (T::PAD == 0 || M::MG % T::RB == 0 || T::RB % M::MG == 0)) {
        // rows of this thread: mr = i*MG + mg for every batch row b -> compile-time offsets from one base
        constexpr int NI = T::Mrow / M::MG;
        const float *xp0 = X + T::roff(mg) + kt * TK;
        const float *yp0 = dY + yoff + ((k == 0) ? mg * KSo : (mg / Jp) * KSo + (mg % Jp) * T::r);
#pragma unroll 1
        for (int b = 0; b < R; ++b) {
#pragma unroll(unroll_of(NI) == NI ? NI : 4)
            for (int i = 0; i < NI; ++i) {
                const int dm = i * M::MG;                                        // compile-time row distance
                const int dy = (k == 0) ? dm * KSo
                                        : ((M::MG % Jp == 0) ? (dm / Jp) * KSo : (dm / Jp) * KSo + (dm % Jp) * T::r);
                row_fma(xp0 + b * T::BS + dm * T::KS + (dm / T::RB) * T::PAD, yp0 + b * BSo + dy);
            }
        }
    } else {
#pragma unroll 2
        for (int it = 0; it < M::ROWS; ++it) {
            const int m = it * M::MG + mg;
            if (M::M % M::MG != 0 && m >= M::M) break;
            const int b = m / T::Mrow, mr = m % T::Mrow;
            row_fma(X + b * T::BS + T::roff(mr) + kt * TK,
                    dY + b * BSo + ((k == 0) ? mr * KSo : (mr / Jp) * KSo + (mr % Jp) * T::r) + yoff);
        }
    }
}

// end of launch: sum the MG row groups of stage k and add the result to the gradient slot
// (blob layout r,i,j,r').  stg: shared staging of K*NS floats (reuses the activation slots).
template <class S, int k, int R, int TK>
TTS_DEV void flush_dw(f32x2 (&acc2)[TK][2], float *__restrict__ stg, float *__restrict__ slot, int tid) {
    using T = St<S, k>;
    float acc[TK][4];
#pragma unroll
    for (int a = 0; a < TK; ++a) {
        upk2(acc2[a][0], acc[a][0], acc[a][1]);
        upk2(acc2[a][1], acc[a][2], acc[a][3]);
    }
    using M = BwMap<S, k, R, TK>;
    constexpr int I0p = T::PACK ? T::I / (T::PACK ? S::G : 1) : 1;
    int nt, kt, mg;
    M::coords(tid, nt, kt, mg);
    __syncthreads();
    for (int g = 0; g < M::MG; ++g) {
        if (mg == g) {
#pragma unroll
            for (int a = 0; a < TK; ++a)
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    float *p = stg + (kt * TK + a) * T::NS + nt * 4 + c;
                    *p = (g == 0) ? acc[a][c] : *p + acc[a][c];
                }
        }
        __syncthreads();
    }
    // staged layout = W_k shared layout [kappa][NS]; scatter-add to the blob
    for (int e = tid; e < T::CORE; e += NTHR) {
        const int ap = e % T::rn;
        int t = e / T::rn;
        const int j = t % T::J;
        t /= T::J;
        const int i = t % T::I;
        const int a = t / T::I;
        const int col = (k == 0 && T::PACK) ? gate_col<S>(i % I0p, i / I0p) : i * T::r + a;
        slot[COff<S, k>::v + e] += stg[(j * T::rn + ap) * T::NS + col];
    }
    __syncthreads();
}

// ---- backward tuning: forward tiles (recompute) + bwd-data tiles + bwd-weight tiles -------------
// BTM[k] rows per thread of the bwd-data stage k, BSP = split of the last bwd-data stage, WTK[k] = TK
template <class FT, int BTM0, int BTM1, int BTM2, int BTM3, int BSP_, int WTK0, int WTK1, int WTK2, int WTK3>
struct TuneB {
    using F = FT;
    static constexpr int BTM[4] = {BTM0, BTM1, BTM2, BTM3};
    static constexpr int BSP = BSP_;
    static constexpr int WTK[4] = {WTK0, WTK1, WTK2, WTK3};
};

// DWI = true : every X_k kept, core gradients accumulated in the recurrent kernel ("fused" backward)
// DWI = false: X_k slots ping-pong like the forward kernel; the kernel only propagates dh/dc and writes
//              delta; the core gradients come from a batched TT-matvec backward over (h_{t-1}, delta)
//              ("split" backward, for chains whose kept slots exceed shared memory)
template <class S, int R, class TB, bool DWI = true, int SV = 0>
struct BwdSmem {
    static constexpr int D = S::D;
    using TU = typename TB::F;
    using FM = FinMap<S, R, TU::FTMr, TU::FTI, TU::FSK>;
    // forward-layout cores are only staged by the kernels that recompute (part of) the chain
    static constexpr int W = (!DWI && SV != 0) ? 0 : w_floats<S>();
    static constexpr int WT = wt_floats<S>();
    static constexpr int stage_bs(int k) { return slot_floats_of<S>(k); }
    static constexpr int HS0 = cr4(R * stage_bs(S::D - 1));
    static constexpr int xoff(int k) {
        if (DWI) {
            int v = 0;
            for (int q = S::D - 1; q > k; --q) v += cr4(R * stage_bs(q));
            return v;
        }
        if (k == S::D - 1) return 0;
        return HS0 + (((S::D - 2 - k) % 2 == 0) ? 0 : PPSlots<S, R>::P);
    }
    template <int k> struct XOff { static constexpr int v = xoff(k); };
    static constexpr int XALL = DWI ? xoff(0) + cr4(R * stage_bs(0)) : HS0 + PPSlots<S, R>::P + PPSlots<S, R>::Q;
    static constexpr int DY = cr4(R * DY0<S>::BS);
    static constexpr int DHC = cr4(R * St<S, D - 1>::BS);
    static constexpr int XCH = cmax(FM::XCH_FLOATS, BdMap<S, D - 1, R, TB::BTM[D - 1], TB::BSP>::XCH_FLOATS);
    static constexpr int H2 = cr4(R * St<S, D - 1>::BS);          // second h_{t-1} slot (cp.async double buffer)
    static constexpr int X1W = (SV != 0) ? 2 * R * XW : 0;        // rank-one input windows (kept-gates kernels)
    static constexpr int DHO = (SV != 0) ? cr4(R * n_in<S>()) : 0; // upstream-gradient tile dOut[:, t, :] (kept-gates kernels)
    static constexpr int TOTAL = W + WT + XALL + DY + DHC + XCH + H2 + X1W + DHO;
    static constexpr size_t BYTES = (size_t)TOTAL * 4;
};

struct RnnBwdSArgs {
    int t0, steps, T;
    long long B;
    float *xg;               // MODE_XG: chunk buffer (B, steps, G*H): ih projection in, delta_ih out
    long long xg_bstride;
    const float *x1;         // MODE_RANK1: x (B, T) (not offset), row stride x1_bstride
    long long x1_bstride;
    const float *w_eff, *bias_ih;
    const float *cores, *bias_hh;
    const float *hs, *cs;    // (B,T,H) outputs / cell states of this layer
    const float *h0, *c0;
    const float *dhs;        // (B,T,H) or null
    const float *dh_in, *dc_in;
    float *dh_out, *dc_out;
    float *partial;          // [gridDim.x][core_floats + 3*G*H]: cores, db_hh, d_weff, db_ih  (+= at the end)
    const float *u_save;     // kept-gates kernels: gate activations written by the forward kernel
    long long u_bstride;     //   (whole sequence, not offset by t0; row stride in floats)
};

// LASTSYNC = false: no barrier after stage 1 (the caller's next phase does not read X_0 and ends with a barrier)
template <class S, int R, class TB, int k, bool DWI = true, bool LASTSYNC = true>
TTS_DEV void fwd_chain_keep(float *xs, const float *hcur, const float *wsm, int tid) {
    if constexpr (k >= 1) {
        using SM = BwdSmem<S, R, TB, DWI>;
        using TU = typename TB::F;
        const float *X = (k == S::D - 1) ? hcur : xs + SM::template XOff<k>::v;
        fwd_stage<S, k, R, TU::TMr[k], TU::TN[k]>(X, wsm + WOff<S, k>::v, xs + SM::template XOff<k - 1>::v, tid);
        if constexpr (k > 1 || LASTSYNC) __syncthreads();
        fwd_chain_keep<S, R, TB, k - 1, DWI, LASTSYNC>(xs, hcur, wsm, tid);
    }
}

// persistent dW register tiles of every stage
template <class S, int R, class TB>
struct DwRegs {
    f32x2 a0[TB::WTK[0]][2];
    f32x2 a1[S::D > 1 ? TB::WTK[S::D > 1 ? 1 : 0] : 1][2];
    f32x2 a2[S::D > 2 ? TB::WTK[S::D > 2 ? 2 : 0] : 1][2];
    f32x2 a3[S::D > 3 ? TB::WTK[S::D > 3 ? 3 : 0] : 1][2];
};

template <class S, int R, class TB, int k, bool WANT_DX = true, bool DWI = true>
TTS_DEV void bwd_chain(float *xs, float *hcur, float *dy0, float *dhc, const float *wt, float *xch,
                       DwRegs<S, R, TB> &dw, int tid) {
    using SM = BwdSmem<S, R, TB, DWI>;
    float *X = (k == S::D - 1) ? hcur : xs + SM::template XOff<k>::v;
    const float *dY = (k == 0) ? dy0 : xs + SM::template XOff<(k == 0 ? 0 : k - 1)>::v;
    if constexpr (DWI && k == 0) bwd_weight_stage<S, 0, R, TB::WTK[0]>(X, dY, dw.a0, tid);
    if constexpr (DWI && k == 1) bwd_weight_stage<S, 1, R, TB::WTK[1]>(X, dY, dw.a1, tid);
    if constexpr (DWI && k == 2) bwd_weight_stage<S, 2, R, TB::WTK[2]>(X, dY, dw.a2, tid);
    if constexpr (DWI && k == 3) bwd_weight_stage<S, 3, R, TB::WTK[3]>(X, dY, dw.a3, tid);
    if constexpr (k == S::D - 1) {
        // last stage: dX goes to the dh slot (no aliasing with X_k); split reduction
        if constexpr (WANT_DX) bwd_data_stage<S, k, R, TB::BTM[k], TB::BSP>(dY, wt + WTOff<S, k>::v, dhc, xch, tid);
        // the cp.async tiles of the NEXT step (h_{t-2}, dOut[:, t-1]) were issued at least one stage ago: waiting for them
        // here lets this barrier also publish them, so the step loop needs no barrier of its own at the top
        cp_async_wait_all();
        __syncthreads();
    } else {
        if constexpr (DWI) __syncthreads();               // X_k is overwritten in place by dX_k
        bwd_data_stage<S, k, R, TB::BTM[k], 1>(dY, wt + WTOff<S, k>::v, X, xch, tid);
        __syncthreads();
        bwd_chain<S, R, TB, k + 1, WANT_DX, DWI>(xs, hcur, dy0, dhc, wt, xch, dw, tid);
    }
}

template <class S, int R, class TB, int k>
TTS_DEV void flush_all(DwRegs<S, R, TB> &dw, float *stg, float *slot, int tid) {
    if constexpr (k == 0) flush_dw<S, 0, R, TB::WTK[0]>(dw.a0, stg, slot, tid);
    if constexpr (k == 1) flush_dw<S, 1, R, TB::WTK[1]>(dw.a1, stg, slot, tid);
    if constexpr (k == 2) flush_dw<S, 2, R, TB::WTK[2]>(dw.a2, stg, slot, tid);
    if constexpr (k == 3) flush_dw<S, 3, R, TB::WTK[3]>(dw.a3, stg, slot, tid);
    if constexpr (k + 1 < S::D) flush_all<S, R, TB, k + 1>(dw, stg, slot, tid);
}

// SV = 0: recompute the whole chain;
// SV = 2: forward kept the hh pre-activations u (G*H floats per row and step): stages d-1..1 are
//         recomputed (their X_k feed the core gradients) but the final stage, its reduce-scatter and two
//         barriers are skipped -- for two-core chains that is 60 % of the recomputed multiply-adds
template <class S, int CELL, int R, int MODE, class TB, bool DWI = true, int SV = 0, int MINB = 1>
__global__ void __launch_bounds__(NTHR, MINB) k_rnn_bwd_s(const __grid_constant__ RnnBwdSArgs a) {
    static_assert(SV == 0 || SV == 2, "save mode");
    constexpr bool SAVEU = (SV != 0);
    static_assert(!SrcOf<S>::merged || (!DWI && SV == 2), "contracted chains run the dX-only kernel with kept gates");
    // DWI = false with kept gates: nothing of the forward chain is needed (gates come from the forward pass, the
    // core gradients from the dense accumulation outside): the kernel runs the gate gradients and the dX chain only
    constexpr bool RECOMPUTE = DWI || !SAVEU;
    constexpr bool NEED_H = DWI || !SAVEU || (CELL != TTRNN_CELL_LSTM);
    extern __shared__ __align__(16) float smem[];
    using SM = BwdSmem<S, R, TB, DWI, SV>;
    // split backward: the kernel writes delta_hh of every step to the xg buffer for the dense accumulation of the hh core
    // gradients.  Projected input (MODE_XG): the same buffer must carry delta_ih, so delta_hh has to equal delta_ih (LSTM).
    // Rank-one input: the ih gradients are accumulated in registers (g_weff / g_bih), the buffer carries delta_hh only.
    static_assert(DWI || MODE == MODE_RANK1 || (CELL == TTRNN_CELL_LSTM && MODE == MODE_XG),
                  "split backward with a projected input needs delta_hh == delta_ih (LSTM)");
    using FM = typename SM::FM;
    using TL = St<S, S::D - 1>;
    using T0 = St<S, 0>;
    constexpr int G = S::G, H = n_in<S>(), GH = G * H;
    constexpr int NE = FM::NE;
    constexpr bool LSTM = (CELL == TTRNN_CELL_LSTM);
    const int tid = threadIdx.x;
    float *wsm = smem;
    float *wt = wsm + SM::W;
    float *xs = wt + SM::WT;
    float *dy0 = xs + SM::XALL;
    float *dhc = dy0 + SM::DY;
    float *xch = dhc + SM::DHC;
    // the two h_{t-1} slots as offsets from the shared base (a pointer array would lose the address space)
    constexpr int HOFF0 = SM::W + SM::WT + SM::template XOff<S::D - 1>::v;
    constexpr int HOFF1 = SM::W + SM::WT + SM::XALL + SM::DY + SM::DHC + SM::XCH;
    float *xw1 = smem + HOFF1 + SM::H2;
    float *dho_s = xw1 + SM::X1W;

    if constexpr (SM::W > 0) stage_weights_k<S, 0>(a.cores, wsm, tid);
    stage_weights_t<S, 0>(a.cores, wt, tid);
    for (int e = tid; e < SM::DY; e += NTHR) dy0[e] = 0.f;       // padded gate column stays zero

    int mt, itg, kh;
    FM::coords(tid, mt, itg, kh);
    int hid[NE];
    float bhh[NE][4], weff[NE][4], bih[NE][4];
    float g_bhh[NE][4], g_weff[NE][4], g_bih[NE][4];             // gradient accumulators (whole launch)
#pragma unroll
    for (int n = 0; n < NE; ++n) {
        hid[n] = FM::hidden(mt, itg, n * FM::SK + kh);
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            const int col = g * H + hid[n];
            const bool ok = g < G;
            bhh[n][g] = (ok && a.bias_hh) ? __ldg(a.bias_hh + col) : 0.f;
            weff[n][g] = (ok && MODE == MODE_RANK1) ? __ldg(a.w_eff + col) : 0.f;
            bih[n][g] = (ok && MODE == MODE_RANK1 && a.bias_ih) ? __ldg(a.bias_ih + col) : 0.f;
            g_bhh[n][g] = 0.f; g_weff[n][g] = 0.f; g_bih[n][g] = 0.f;
        }
    }
    DwRegs<S, R, TB> dw;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
#pragma unroll
        for (int q = 0; q < (int)(sizeof(dw.a0) / 16); ++q) dw.a0[q][c] = 0ull;
#pragma unroll
        for (int q = 0; q < (int)(sizeof(dw.a1) / 16); ++q) dw.a1[q][c] = 0ull;
#pragma unroll
        for (int q = 0; q < (int)(sizeof(dw.a2) / 16); ++q) dw.a2[q][c] = 0ull;
#pragma unroll
        for (int q = 0; q < (int)(sizeof(dw.a3) / 16); ++q) dw.a3[q][c] = 0ull;
    }

    const long long ntiles = (a.B + R - 1) / R;
    for (long long tile_i = blockIdx.x; tile_i < ntiles; tile_i += gridDim.x) {
        const long long row0 = tile_i * R;
        __syncthreads();
        for (int e = tid; e < SM::DHC; e += NTHR) dhc[e] = 0.f;
        float dhd[R][NE], dcs[R][NE];                            // direct dh term (GRU) and dc, per owned unit
#pragma unroll
        for (int b = 0; b < R; ++b)
#pragma unroll
            for (int n = 0; n < NE; ++n) {
                const bool ok = row0 + b < a.B;
                dhd[b][n] = (ok && a.dh_in) ? __ldg(a.dh_in + (row0 + b) * H + hid[n]) : 0.f;
                dcs[b][n] = (LSTM && ok && a.dc_in) ? __ldg(a.dc_in + (row0 + b) * H + hid[n]) : 0.f;
            }
        const int nvalid = (a.B - row0 < R) ? (int)(a.B - row0) : R;
        const float *us_p[NE], *cs_p[NE];                 // per-unit bases of the kept gate activations / cell states
#pragma unroll
        for (int n = 0; n < NE; ++n) {
            us_p[n] = a.u_save ? a.u_save + row0 * a.u_bstride + 4 * hid[n] : nullptr;
            cs_p[n] = (LSTM && a.cs) ? a.cs + row0 * (long long)a.T * H + hid[n] : nullptr;
        }
        // h_{t-1} tiles are double-buffered with cp.async one step ahead; per-unit operands of the gate
        // phase are fetched into registers one step ahead as well
        auto fetch_h = [&](float *dst, int tgl) {          // h_{tgl-1} -> dst (X_{d-1} layout)
            for (int e = tid * 4; e < R * H; e += NTHR * 4) {
                const int b = e / H, h = e % H;
                const long long row = row0 + b;
                float *d4 = dst + b * TL::BS + (h / TL::K) * TL::KS + (h % TL::K);
                const float *src = nullptr;
                if (row < a.B) {
                    if (tgl > 0) src = a.hs + (row * a.T + (tgl - 1)) * H + h;
                    else if (a.h0) src = a.h0 + row * H + h;
                }
                if (src) cp_async16(d4, src);
                else st4(d4, make_float4(0.f, 0.f, 0.f, 0.f));
            }
        };
        // Recompute kernels (SV = 0) fetch the per-unit operands of the gate phase into registers one step ahead.
        // The kept-gates kernels (SV != 0) instead read this step's gate activations / c_{t-1} at the top of the
        // step (they are consumed after the chain recompute), take x[b, t] from the shared windows and the
        // upstream gradient from a cp.async tile: no value is carried across steps in registers, which at 255
        // registers per thread were being spilled (and a spilled prefetch waits for its own load).
        float xin_n[R][NE][4], x1_n[R], cprev_n[R][NE], dho_n[R][NE];
        auto fetch_dho = [&](int tgl) {                   // dOut[:, tgl, :] of the CTA's rows -> dho_s [b][h]
            for (int e = tid * 4; e < R * H; e += NTHR * 4) {
                const int b = e / H, h = e % H;
                const long long row = row0 + b;
                if (row < a.B && a.dhs) cp_async16(dho_s + e, a.dhs + (row * a.T + tgl) * H + h);
                else st4(dho_s + e, make_float4(0.f, 0.f, 0.f, 0.f));
            }
        };
        auto fetch_regs = [&](int tl) {                   // operands of local step tl (recompute kernels)
            const int tgl = a.t0 + tl;
#pragma unroll
            for (int b = 0; b < R; ++b) {
                const long long row = row0 + b;
                const bool ok = row < a.B;
                x1_n[b] = (MODE == MODE_RANK1 && ok) ? __ldg(a.x1 + row * a.x1_bstride + tgl) : 0.f;
#pragma unroll
                for (int n = 0; n < NE; ++n) {
                    if (MODE == MODE_XG) {
#pragma unroll
                        for (int g = 0; g < G; ++g)
                            xin_n[b][n][g] = ok ? a.xg[row * a.xg_bstride + (long long)tl * GH + g * H + hid[n]] : 0.f;
                    }
                    float cv = 0.f;
                    if (LSTM && ok) {
                        if (tgl > 0) cv = __ldg(a.cs + (row * a.T + (tgl - 1)) * H + hid[n]);
                        else if (a.c0) cv = __ldg(a.c0 + row * H + hid[n]);
                    }
                    cprev_n[b][n] = cv;
                    dho_n[b][n] = (ok && a.dhs) ? __ldg(a.dhs + (row * a.T + tgl) * H + hid[n]) : 0.f;
                }
            }
        };
        // kept gate activations (LSTM i,f,g,o; GRU r,z,n,u_n) and c_{t-1} of global step tgl
        auto load_kept = [&](int tgl, float (&P)[R][NE][4], float (&Cp)[R][NE]) {
#pragma unroll
            for (int b = 0; b < R; ++b) {
                const bool ok = b < nvalid;
#pragma unroll
                for (int n = 0; n < NE; ++n) {
                    const float4 kv = ok ? __ldg(reinterpret_cast<const float4 *>(us_p[n] + (long long)tgl * (4 * H) + b * a.u_bstride))
                                         : make_float4(0.f, 0.f, 0.f, 0.f);
                    P[b][n][0] = kv.x; P[b][n][1] = kv.y; P[b][n][2] = kv.z; P[b][n][3] = kv.w;
                    float cv = 0.f;
                    if (LSTM && ok) {
                        if (tgl > 0) cv = __ldg(cs_p[n] + (long long)(tgl - 1) * H + (long long)b * a.T * H);
                        else if (a.c0) cv = __ldg(a.c0 + (row0 + b) * H + hid[n]);
                    }
                    Cp[b][n] = cv;
                }
            }
        };
        // dX-only kernels have no recompute phase to hide the latency of these loads behind, and registers to
        // spare: they fetch them one step ahead (ncu: 14 % of the samples sat on the first use of the gates)
        constexpr bool AHEAD = SAVEU && !RECOMPUTE;
        float pre_a[R][NE][4], cprev_a[R][NE];
        if constexpr (AHEAD) load_kept(a.t0 + a.steps - 1, pre_a, cprev_a);
        if constexpr (NEED_H) fetch_h(smem + (((a.steps - 1) & 1) ? HOFF1 : HOFF0), a.t0 + a.steps - 1);
        if constexpr (SAVEU) {
            fetch_dho(a.t0 + a.steps - 1);
            if (MODE == MODE_RANK1) {
                const int wl = (a.steps - 1) / XW;
                x1_fetch_window<R>(xw1 + (wl & 1) * R * XW, a.x1 + a.t0, a.x1_bstride, row0, a.B, a.steps, wl, tid);
                if (wl >= 1)
                    x1_fetch_window<R>(xw1 + ((wl - 1) & 1) * R * XW, a.x1 + a.t0, a.x1_bstride, row0, a.B, a.steps, wl - 1, tid);
            }
        } else {
            fetch_regs(a.steps - 1);
        }
        cp_async_wait_all();
        __syncthreads();
        for (int t = a.steps - 1; t >= 0; --t) {
            const int tg = a.t0 + t;
            float *hcur = smem + ((t & 1) ? HOFF1 : HOFF0);
            // the last barrier of the previous step's backward chain already ordered everything this step reads (dh chain,
            // cp.async tiles)
            // operands of this step
            float xin[R][NE][4], x1[R], cprev[R][NE], hprev[R][NE], dho[R][NE], pre[R][NE][4];
#pragma unroll
            for (int b = 0; b < R; ++b) {
                if constexpr (SAVEU) x1[b] = (MODE == MODE_RANK1) ? xw1[((t / XW) & 1) * R * XW + b * XW + (t % XW)] : 0.f;
                else x1[b] = x1_n[b];
#pragma unroll
                for (int n = 0; n < NE; ++n) {
                    if constexpr (SAVEU) {
                        if constexpr (AHEAD) {
#pragma unroll
                            for (int g = 0; g < 4; ++g) pre[b][n][g] = pre_a[b][n][g];
                            cprev[b][n] = cprev_a[b][n];
                        }
                        dho[b][n] = dho_s[b * H + hid[n]];
                    } else {
#pragma unroll
                        for (int g = 0; g < 4; ++g) xin[b][n][g] = xin_n[b][n][g];
                        cprev[b][n] = cprev_n[b][n];
                        dho[b][n] = dho_n[b][n];
                    }
                    hprev[b][n] = hcur[b * TL::BS + (hid[n] / TL::K) * TL::KS + (hid[n] % TL::K)];
                }
            }
            if constexpr (SAVEU && !AHEAD) load_kept(tg, pre, cprev);   // consumed after the recompute phase
            // request the operands of step t-1 now; they land while this step computes
            if (t > 0) {
                if constexpr (NEED_H) fetch_h(smem + (((t - 1) & 1) ? HOFF1 : HOFF0), tg - 1);
                if constexpr (!SAVEU) fetch_regs(t - 1);
                if constexpr (AHEAD) load_kept(tg - 1, pre_a, cprev_a);
            }
            if constexpr (SAVEU) {
                // entering window w = t / XW from above: stage window w - 1 (its buffer was last read a step ago)
                if (MODE == MODE_RANK1 && (t % XW) == XW - 1 && t != a.steps - 1 && t / XW >= 1)
                    x1_fetch_window<R>(xw1 + ((t / XW - 1) & 1) * R * XW, a.x1 + a.t0, a.x1_bstride, row0, a.B, a.steps,
                                       t / XW - 1, tid);
            }
            // ---- recompute the hh chain keeping every X_k
            // kept-gates kernels: the gate phase below reads neither X_0 nor anything stage 1 writes, so there is
            // no barrier between them -- warps still in stage 1 (FFMA2-bound) overlap with warps already in the
            // latency-bound gate phase; the barrier after the gate phase orders X_0 / dY_0 for the backward chain
            if constexpr (RECOMPUTE) fwd_chain_keep<S, R, TB, S::D - 1, DWI, !SAVEU>(xs, hcur, wsm, tid);
            if constexpr (!SAVEU) {
                float acc[R][FM::TMr][FM::TI][4];
                final_partial<S, R, FM>((S::D == 1) ? hcur : xs + SM::template XOff<0>::v, wsm + WOff<S, 0>::v, mt, itg,
                                        kh, acc);
                final_reduce<S, R, FM>(acc, pre, xch, tid, kh);
            }
            // ---- gates and their gradients
#pragma unroll
            for (int b = 0; b < R; ++b)
#pragma unroll
                for (int n = 0; n < NE; ++n) {
                    const int h = hid[n];
                    const long long row = row0 + b;
                    const bool ok = b < nvalid;
                    float ain[4];
#pragma unroll
                    for (int g = 0; g < G; ++g)
                        ain[g] = SAVEU ? 0.f : ((MODE == MODE_XG) ? xin[b][n][g] : fmaf(x1[b], weff[n][g], bih[n][g]));
                    const float dh = dhd[b][n] + dhc[b * TL::BS + (h / TL::K) * TL::KS + (h % TL::K)] + dho[b][n];
                    float d_ih[4], d_hh[4];
                    d_ih[3] = 0.f; d_hh[3] = 0.f;
                    if (LSTM) {
                        // kept-gates kernels: the activations come from the forward pass, no transcendentals but tanh(c_t)
                        const float ig = SAVEU ? pre[b][n][0] : sigmoidf_acc(pre[b][n][0] + bhh[n][0] + ain[0]);
                        const float fg = SAVEU ? pre[b][n][1] : sigmoidf_acc(pre[b][n][1] + bhh[n][1] + ain[1]);
                        const float gg = SAVEU ? pre[b][n][2] : tanh_g(pre[b][n][2] + bhh[n][2] + ain[2]);
                        const float og = SAVEU ? pre[b][n][3] : sigmoidf_acc(pre[b][n][3] + bhh[n][3] + ain[3]);
                        const float cn = fg * cprev[b][n] + ig * gg;
                        const float tc = tanh_g(cn);
                        const float dc = dcs[b][n] + dh * og * (1.0f - tc * tc);
                        d_hh[0] = dc * gg * ig * (1.0f - ig);
                        d_hh[1] = dc * cprev[b][n] * fg * (1.0f - fg);
                        d_hh[2] = dc * ig * (1.0f - gg * gg);
                        d_hh[3] = dh * tc * og * (1.0f - og);
                        dcs[b][n] = dc * fg;
                        dhd[b][n] = 0.f;
#pragma unroll
                        for (int g = 0; g < 4; ++g) d_ih[g] = d_hh[g];
                    } else {
                        const float ur = pre[b][n][0] + bhh[n][0];
                        const float uz = pre[b][n][1] + bhh[n][1];
                        const float un = SAVEU ? pre[b][n][3] : pre[b][n][2] + bhh[n][2];
                        const float rg = SAVEU ? pre[b][n][0] : sigmoidf_acc(ain[0] + ur);
                        const float zg = SAVEU ? pre[b][n][1] : sigmoidf_acc(ain[1] + uz);
                        const float ng = SAVEU ? pre[b][n][2] : tanh_g(ain[2] + rg * un);
                        const float d_n = dh * (1.0f - zg) * (1.0f - ng * ng);
                        const float d_z = dh * (hprev[b][n] - ng) * zg * (1.0f - zg);
                        const float d_r = d_n * un * rg * (1.0f - rg);
                        d_ih[0] = d_r; d_ih[1] = d_z; d_ih[2] = d_n;
                        d_hh[0] = d_r; d_hh[1] = d_z; d_hh[2] = d_n * rg;
                        dhd[b][n] = dh * zg;
                    }
                    if (!ok) {
#pragma unroll
                        for (int g = 0; g < 4; ++g) { d_ih[g] = 0.f; d_hh[g] = 0.f; }
                    }
                    // delta_hh -> dY_0 [b][mr][i0'*4 + g]
                    const int mr = h % T0::Mrow, i0p = h / T0::Mrow;
                    float *dyr = dy0 + b * DY0<S>::BS + mr * DY0<S>::DS;
                    if (G == 4) {
                        st4(dyr + i0p * 4, make_float4(d_hh[0], d_hh[1], d_hh[2], d_hh[3]));
                    } else {
                        *reinterpret_cast<float2 *>(dyr + gate_col<S>(i0p, 0)) = make_float2(d_hh[0], d_hh[1]);
                        dyr[gate_col<S>(i0p, 2)] = d_hh[2];
                    }
#pragma unroll
                    for (int g = 0; g < G; ++g) {
                        if (MODE == MODE_RANK1) {
                            g_weff[n][g] = fmaf(d_ih[g], x1[b], g_weff[n][g]);
                            g_bih[n][g] += d_ih[g];
                            if (!DWI && ok) a.xg[row * a.xg_bstride + (long long)t * GH + g * H + h] = d_hh[g];
                        } else if (ok) {
                            a.xg[row * a.xg_bstride + (long long)t * GH + g * H + h] = d_ih[g];
                        }
                        g_bhh[n][g] += d_hh[g];
                    }
                }
            __syncthreads();
            if constexpr (SAVEU) {
                if (t > 0) fetch_dho(tg - 1);             // the tile of this step has been consumed by every thread
            }
            // ---- backward chain: core gradients (register tiles) and dh_{t-1}
            bwd_chain<S, R, TB, 0, true, DWI>(xs, hcur, dy0, dhc, wt, xch, dw, tid);
            cp_async_wait_all();
        }
        __syncthreads();
#pragma unroll
        for (int b = 0; b < R; ++b)
#pragma unroll
            for (int n = 0; n < NE; ++n)
                if (row0 + b < a.B) {
                    const int h = hid[n];
                    a.dh_out[(row0 + b) * H + h] = dhd[b][n] + dhc[b * TL::BS + (h / TL::K) * TL::KS + (h % TL::K)];
                    if (LSTM) a.dc_out[(row0 + b) * H + h] = dcs[b][n];
                }
    }
    // ---- flush gradients of this CTA into its slot
    if (!a.partial) return;
    float *slot = a.partial + (long long)blockIdx.x * (blob_floats<S>() + 3 * GH);
    if constexpr (DWI) flush_all<S, R, TB, 0>(dw, xs, slot, tid);
#pragma unroll
    for (int n = 0; n < NE; ++n)
#pragma unroll
        for (int g = 0; g < G; ++g) {
            const int col = g * H + hid[n];
            slot[blob_floats<S>() + col] += g_bhh[n][g];
            slot[blob_floats<S>() + GH + col] += g_weff[n][g];
            slot[blob_floats<S>() + 2 * GH + col] += g_bih[n][g];
        }
}

// =============================================================================================
// Batched TT matvec (ih projection of a time chunk, stand-alone TTLinear) -- static path
// Shapes have G = 0 (plain stage-0 layout).  Rows are processed in tiles of R; CTAs are persistent.
// =============================================================================================
template <class S, int R, int TMr_>
struct OutMap {
    using T = St<S, 0>;
    static_assert(T::r == 1 && (T::N == 4 || T::N == 8), "output stage handles a first mode of 4 or 8");
    static constexpr int TMr = TMr_, TN = T::N;
    static constexpr int MTl = T::Mrow / TMr;
    static_assert(T::Mrow % TMr == 0 && NTHR % MTl == 0 && MTl % 32 == 0, "output stage tile grid");
    static constexpr int RB = NTHR / MTl;                // groups of threads that split the R batch rows
    static constexpr int RPT = (R + RB - 1) / RB;        // batch rows per thread
};

struct TtlFwdSArgs {
    long long rows;
    int rows_per_b;
    long long x_bstride, y_bstride;
    const float *x, *cores, *bias, *bias2;
    float *y;
};

template <class S, int R, class TU>
struct TtlFwdSmem {
    static constexpr int W = w_floats<S>();
    static constexpr int HS = cr4(R * St<S, S::D - 1>::BS);
    static constexpr int P = PPSlots<S, R>::P, Q = PPSlots<S, R>::Q;
    static constexpr int TOTAL = W + HS + P + Q;
    static constexpr size_t BYTES = (size_t)TOTAL * 4;
};

// rows (global) -> X_{d-1} slot; pad columns of the slot are zeroed once by the caller
template <class S, int R>
TTS_DEV void load_rows(const float *__restrict__ x, long long row0, long long rows, int rows_per_b, long long bstride,
                       float *__restrict__ slot, int tid) {
    using TL = St<S, S::D - 1>;
    constexpr int NIN = n_in<S>();
    for (int e = tid; e < R * NIN; e += NTHR) {
        const int b = e / NIN, c = e % NIN;
        const long long row = row0 + b;
        float v = 0.f;
        if (row < rows) {
            const long long bb = row / rows_per_b, tt = row - bb * rows_per_b;
            v = __ldg(x + bb * bstride + tt * NIN + c);
        }
        slot[b * TL::BS + (c / TL::Kraw) * TL::KS + (c % TL::Kraw)] = v;
    }
}

template <class S, int R, class TU>
__global__ void __launch_bounds__(NTHR, 1) k_ttlin_fwd_s(const __grid_constant__ TtlFwdSArgs a) {
    extern __shared__ __align__(16) float smem[];
    using SM = TtlFwdSmem<S, R, TU>;
    using T0 = St<S, 0>;
    using OM = OutMap<S, R, TU::FTMr>;
    constexpr int NOUT = n_out<S>();
    const int tid = threadIdx.x;
    float *wsm = smem;
    float *hs = wsm + SM::W;
    float *P = hs + SM::HS;
    float *Q = P + SM::P;
    stage_weights_k<S, 0>(a.cores, wsm, tid);
    for (int e = tid; e < SM::HS; e += NTHR) hs[e] = 0.f;
    const int mt = tid % OM::MTl, rb = tid / OM::MTl;
    // bias of the columns this thread writes: col(j, q) = j*Mrow_0 + q*MTl + mt
    float bias[OM::TMr][OM::TN];
#pragma unroll
    for (int q = 0; q < OM::TMr; ++q)
#pragma unroll
        for (int j = 0; j < OM::TN; ++j) {
            const int col = j * T0::Mrow + q * OM::MTl + mt;
            bias[q][j] = (a.bias ? __ldg(a.bias + col) : 0.f) + (a.bias2 ? __ldg(a.bias2 + col) : 0.f);
        }
    const long long ntiles = (a.rows + R - 1) / R;
    for (long long tile_i = blockIdx.x; tile_i < ntiles; tile_i += gridDim.x) {
        const long long row0 = tile_i * R;
        __syncthreads();
        load_rows<S, R>(a.x, row0, a.rows, a.rows_per_b, a.x_bstride, hs, tid);
        __syncthreads();
        const float *X0 = fwd_chain_pp<S, R, TU, S::D - 1>(hs, P, Q, wsm, tid);
        // ---- output stage: thread = (row tile mt, batch-row group rb); lanes run along rows, so every
        // global store of a warp covers 32 consecutive floats
        float acc[OM::RPT][OM::TMr][OM::TN];
        f32x2 acc2[OM::RPT][OM::TMr][OM::TN / 2];
#pragma unroll
        for (int i = 0; i < OM::RPT; ++i)
#pragma unroll
            for (int q = 0; q < OM::TMr; ++q)
#pragma unroll
                for (int j = 0; j < OM::TN / 2; ++j) acc2[i][q][j] = 0ull;
        const float *xb = X0 + T0::roff(mt);
        const float *wb = wsm + WOff<S, 0>::v;
#pragma unroll 2
        for (int k4 = 0; k4 < T0::K; k4 += 4) {
            float4 av[OM::RPT][OM::TMr];
#pragma unroll
            for (int i = 0; i < OM::RPT; ++i)
#pragma unroll
                for (int q = 0; q < OM::TMr; ++q) {
                    const int b = rb * OM::RPT + i;
                    av[i][q] = ld4(xb + (b < R ? b : 0) * T0::BS + (T0::roff(mt + q * OM::MTl) - T0::roff(mt)) + k4);
                }
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                f32x2 w2[OM::TN / 2];
#pragma unroll
                for (int g = 0; g < OM::TN / 4; ++g) {
                    const float4 t = ld4(wb + (k4 + kk) * T0::NS + 4 * g);
                    w2[2 * g] = pk2(t.x, t.y);
                    w2[2 * g + 1] = pk2(t.z, t.w);
                }
#pragma unroll
                for (int i = 0; i < OM::RPT; ++i)
#pragma unroll
                    for (int q = 0; q < OM::TMr; ++q) {
                        const float x = kk == 0 ? av[i][q].x : (kk == 1 ? av[i][q].y : (kk == 2 ? av[i][q].z : av[i][q].w));
#pragma unroll
                        for (int j = 0; j < OM::TN / 2; ++j) ffma2(acc2[i][q][j], x, w2[j]);
                    }
            }
        }
#pragma unroll
        for (int i = 0; i < OM::RPT; ++i)
#pragma unroll
            for (int q = 0; q < OM::TMr; ++q)
#pragma unroll
                for (int j = 0; j < OM::TN / 2; ++j) upk2(acc2[i][q][j], acc[i][q][2 * j], acc[i][q][2 * j + 1]);
#pragma unroll
        for (int i = 0; i < OM::RPT; ++i) {
            const int b = rb * OM::RPT + i;
            const long long row = row0 + b;
            if (b < R && row < a.rows) {
                const long long bb = row / a.rows_per_b, tt = row - bb * a.rows_per_b;
                float *yr = a.y + bb * a.y_bstride + tt * NOUT;
#pragma unroll
                for (int q = 0; q < OM::TMr; ++q)
#pragma unroll
                    for (int j = 0; j < OM::TN; ++j) yr[j * T0::Mrow + q * OM::MTl + mt] = acc[i][q][j] + bias[q][j];
            }
        }
    }
}

// ---- backward of the batched TT matvec ---------------------------------------------------------
template <bool W, class S, int k, int R, int TM, int SP> struct XchSel { static constexpr int v = 0; };
template <class S, int k, int R, int TM, int SP> struct XchSel<true, S, k, R, TM, SP> {
    static constexpr int v = BdMap<S, k, R, TM, SP>::XCH_FLOATS;
};

struct TtlBwdSArgs {
    long long rows;
    int rows_per_b;
    long long x_bstride, dy_bstride, dx_bstride;
    const float *x, *cores, *dy;
    float *dx;               // used only by the WANT_DX instantiation
    float *partial;          // [gridDim.x][core_floats + n_out]
    int want_dbias;
};

template <class S, int R, class TB, bool WANT_DX>
struct TtlBwdSmem {
    static constexpr int W = w_floats<S>();
    static constexpr int WT = wt_floats<S>();
    static constexpr int stage_bs(int k) { return slot_floats_of<S>(k); }
    static constexpr int xoff(int k) {
        int v = 0;
        for (int q = S::D - 1; q > k; --q) v += cr4(R * stage_bs(q));
        return v;
    }
    template <int k> struct XOff { static constexpr int v = xoff(k); };
    static constexpr int XALL = xoff(0) + cr4(R * stage_bs(0));
    static constexpr int DY = cr4(R * DY0<S>::BS);
    static constexpr int DXS = WANT_DX ? cr4(R * St<S, S::D - 1>::BS) : 0;
    static constexpr int XCH = XchSel<WANT_DX, S, S::D - 1, R, TB::BTM[S::D - 1], TB::BSP>::v;
    static constexpr int TOTAL = W + WT + XALL + DY + DXS + XCH;
    static constexpr size_t BYTES = (size_t)TOTAL * 4;
};

template <class S, int R, class TB, int k, class SM>
TTS_DEV void ttl_fwd_keep(float *xs, const float *wsm, int tid) {
    if constexpr (k >= 1) {
        using TU = typename TB::F;
        fwd_stage<S, k, R, TU::TMr[k], TU::TN[k]>(xs + SM::template XOff<k>::v, wsm + WOff<S, k>::v,
                                                   xs + SM::template XOff<k - 1>::v, tid);
        __syncthreads();
        ttl_fwd_keep<S, R, TB, k - 1, SM>(xs, wsm, tid);
    }
}

template <class S, int R, class TB, int k, bool WANT_DX, class SM>
TTS_DEV void ttl_bwd_chain(float *xs, float *dy0, float *dxs, const float *wt, float *xch, DwRegs<S, R, TB> &dw, int tid) {
    float *X = xs + SM::template XOff<k>::v;
    const float *dY = (k == 0) ? dy0 : xs + SM::template XOff<(k == 0 ? 0 : k - 1)>::v;
    if constexpr (k == 0) bwd_weight_stage<S, 0, R, TB::WTK[0]>(X, dY, dw.a0, tid);
    if constexpr (k == 1) bwd_weight_stage<S, 1, R, TB::WTK[1]>(X, dY, dw.a1, tid);
    if constexpr (k == 2) bwd_weight_stage<S, 2, R, TB::WTK[2]>(X, dY, dw.a2, tid);
    if constexpr (k == 3) bwd_weight_stage<S, 3, R, TB::WTK[3]>(X, dY, dw.a3, tid);
    if constexpr (k == S::D - 1) {
        if constexpr (WANT_DX) bwd_data_stage<S, k, R, TB::BTM[k], TB::BSP>(dY, wt + WTOff<S, k>::v, dxs, xch, tid);
        __syncthreads();
    } else {
        __syncthreads();
        bwd_data_stage<S, k, R, TB::BTM[k], 1>(dY, wt + WTOff<S, k>::v, X, xch, tid);
        __syncthreads();
        ttl_bwd_chain<S, R, TB, k + 1, WANT_DX, SM>(xs, dy0, dxs, wt, xch, dw, tid);
    }
}

template <class S, int R, class TB, bool WANT_DX>
__global__ void __launch_bounds__(NTHR, 1) k_ttlin_bwd_s(const __grid_constant__ TtlBwdSArgs a) {
    extern __shared__ __align__(16) float smem[];
    using SM = TtlBwdSmem<S, R, TB, WANT_DX>;
    using T0 = St<S, 0>;
    using TL = St<S, S::D - 1>;
    constexpr int NOUT = n_out<S>(), NIN = n_in<S>();
    static_assert(NOUT % NTHR == 0, "bias-gradient ownership needs n_out to be a multiple of the block size");
    constexpr int CPT = NOUT / NTHR;                      // output columns owned per thread (bias gradient)
    const int tid = threadIdx.x;
    float *wsm = smem;
    float *wt = wsm + SM::W;
    float *xs = wt + SM::WT;
    float *dy0 = xs + SM::XALL;
    float *dxs = dy0 + SM::DY;
    float *xch = dxs + SM::DXS;
    stage_weights_k<S, 0>(a.cores, wsm, tid);
    stage_weights_t<S, 0>(a.cores, wt, tid);
    for (int e = tid; e < cr4(R * TL::BS); e += NTHR) xs[SM::template XOff<S::D - 1>::v + e] = 0.f;
    float dbias[CPT];
#pragma unroll
    for (int j = 0; j < CPT; ++j) dbias[j] = 0.f;
    DwRegs<S, R, TB> dw;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
#pragma unroll
        for (int q = 0; q < (int)(sizeof(dw.a0) / 16); ++q) dw.a0[q][c] = 0ull;
#pragma unroll
        for (int q = 0; q < (int)(sizeof(dw.a1) / 16); ++q) dw.a1[q][c] = 0ull;
#pragma unroll
        for (int q = 0; q < (int)(sizeof(dw.a2) / 16); ++q) dw.a2[q][c] = 0ull;
#pragma unroll
        for (int q = 0; q < (int)(sizeof(dw.a3) / 16); ++q) dw.a3[q][c] = 0ull;
    }
    const long long ntiles = (a.rows + R - 1) / R;
    for (long long tile_i = blockIdx.x; tile_i < ntiles; tile_i += gridDim.x) {
        const long long row0 = tile_i * R;
        __syncthreads();
        load_rows<S, R>(a.x, row0, a.rows, a.rows_per_b, a.x_bstride, xs + SM::template XOff<S::D - 1>::v, tid);
        // dy rows -> dY_0 [b][mr][i0]; the thread that reads column c also owns its bias gradient
#pragma unroll
        for (int j = 0; j < CPT; ++j) {
            const int c = tid + j * NTHR;
            const int i0 = c / T0::Mrow, mr = c % T0::Mrow;
#pragma unroll
            for (int b = 0; b < R; ++b) {
                const long long row = row0 + b;
                float v = 0.f;
                if (row < a.rows) {
                    const long long bb = row / a.rows_per_b, tt = row - bb * a.rows_per_b;
                    v = __ldg(a.dy + bb * a.dy_bstride + tt * NOUT + c);
                }
                dy0[b * DY0<S>::BS + mr * DY0<S>::DS + i0] = v;
                dbias[j] += v;
            }
        }
        __syncthreads();
        ttl_fwd_keep<S, R, TB, S::D - 1, SM>(xs, wsm, tid);
        ttl_bwd_chain<S, R, TB, 0, WANT_DX, SM>(xs, dy0, dxs, wt, xch, dw, tid);
        if constexpr (WANT_DX) {
            for (int e = tid; e < R * NIN; e += NTHR) {
                const int b = e / NIN, c = e % NIN;
                const long long row = row0 + b;
                if (row < a.rows) {
                    const long long bb = row / a.rows_per_b, tt = row - bb * a.rows_per_b;
                    a.dx[bb * a.dx_bstride + tt * NIN + c] = dxs[b * TL::BS + (c / TL::Kraw) * TL::KS + (c % TL::Kraw)];
                }
            }
        }
    }
    float *slot = a.partial + (long long)blockIdx.x * (core_floats<S>() + NOUT);
    flush_all<S, R, TB, 0>(dw, xs, slot, tid);
    if (a.want_dbias) {
#pragma unroll
        for (int j = 0; j < CPT; ++j) slot[core_floats<S>() + tid + j * NTHR] += dbias[j];
    }
}

}  // namespace tts
