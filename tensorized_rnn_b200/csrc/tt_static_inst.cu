// Instantiations of the static kernels for the benchmark shapes (BASELINE.json configs 1-5) and the
// lookup used by the C ABI.  Adding a shape = one TTS_SHAPE line + one TTS_FWD line per variant.
#include "tt_static.cuh"
#include "tt_static_api.h"
#include <cstdio>

namespace {

#define TTS_SHAPE(NAME, D_, G_, ...)                          \
    struct NAME {                                             \
        static constexpr int D = D_, G = G_;                  \
        __VA_ARGS__                                           \
    };
#define ARR(name, ...) static constexpr int name[7] = {__VA_ARGS__};

// hidden-to-hidden chains: J = in modes, I = out modes (gates folded into I[0]), RK = ranks r_0..r_d
TTS_SHAPE(HH_H256_d2r4_lstm, 2, 4, ARR(J, 16, 16) ARR(I, 32, 32) ARR(RK, 1, 4, 1))
TTS_SHAPE(HH_H256_d2r4_gru, 2, 3, ARR(J, 16, 16) ARR(I, 24, 32) ARR(RK, 1, 4, 1))
TTS_SHAPE(HH_H256_d3r8_lstm, 3, 4, ARR(J, 4, 8, 8) ARR(I, 8, 8, 16) ARR(RK, 1, 8, 8, 1))
TTS_SHAPE(HH_H256_d4r16_lstm, 4, 4, ARR(J, 4, 4, 4, 4) ARR(I, 4, 4, 8, 8) ARR(RK, 1, 16, 16, 16, 1))
// H = 768 (the reference's default GE2E width, encoder/params_model.py:3; n_cores 2, rank 2 -> rank-padded to 4)
TTS_SHAPE(HH_H768_d2r4_lstm, 2, 4, ARR(J, 24, 32) ARR(I, 48, 64) ARR(RK, 1, 4, 1))
TTS_SHAPE(HH_H1024_d4r8_lstm, 4, 4, ARR(J, 4, 4, 8, 8) ARR(I, 8, 8, 8, 8) ARR(RK, 1, 8, 8, 8, 1))

constexpr size_t kMaxSmem = 232448;     // 227 KB opt-in limit per CTA on sm_100

// input-to-hidden chains (G = 0: plain stage-0 layout); a last in-mode of 5 is zero-padded to 8
TTS_SHAPE(IH_40_H256_d3r8, 3, 0, ARR(J, 2, 4, 5) ARR(I, 8, 8, 16) ARR(RK, 1, 8, 8, 1))
TTS_SHAPE(IH_256_H256_d3r8, 3, 0, ARR(J, 4, 8, 8) ARR(I, 8, 8, 16) ARR(RK, 1, 8, 8, 1))
TTS_SHAPE(IH_256_H1024_d4r8, 4, 0, ARR(J, 4, 4, 4, 4) ARR(I, 8, 8, 8, 8) ARR(RK, 1, 8, 8, 8, 1))
TTS_SHAPE(HHW_H1024_d4r8, 4, 0, ARR(J, 4, 4, 8, 8) ARR(I, 8, 8, 8, 8) ARR(RK, 1, 8, 8, 8, 1))
TTS_SHAPE(IH_40_H256_d4r16, 4, 0, ARR(J, 2, 2, 2, 5) ARR(I, 4, 4, 8, 8) ARR(RK, 1, 16, 16, 16, 1))
TTS_SHAPE(IH_256_H256_d4r16, 4, 0, ARR(J, 4, 4, 4, 4) ARR(I, 4, 4, 8, 8) ARR(RK, 1, 16, 16, 16, 1))

template <class S>
bool match_shape(const ttrnn_tt_shape *s) {
    if (s->d != S::D) return false;
    for (int k = 0; k < S::D; ++k)
        if (s->in_modes[k] != S::J[k] || s->out_modes[k] != S::I[k] || s->ranks[k] != S::RK[k]) return false;
    return s->ranks[S::D] == 1;
}

template <class S, int CELL, int R, int MODE, class TU, int MINB = 1>
int launch_fwd(const tts::RnnFwdSArgs *a, int grid, cudaStream_t st) {
    tts::k_rnn_fwd_s<S, CELL, R, MODE, TU, MINB><<<grid, tts::NTHR, tts::FwdSmem<S, R, TU>::BYTES, st>>>(*a);
    return (int)cudaGetLastError();
}
template <class S, int CELL, int R, int MODE, class TU, int MINB = 1>
int prepare_fwd(int *occ) {
    auto k = tts::k_rnn_fwd_s<S, CELL, R, MODE, TU, MINB>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tts::FwdSmem<S, R, TU>::BYTES);
    if (e != cudaSuccess) return (int)e;
    return (int)cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, k, tts::NTHR, tts::FwdSmem<S, R, TU>::BYTES);
}

#define TTS_FWD(S, CELL, R, MODE, ...)                                                                     \
    {#S, CELL, MODE, R, tts::FwdSmem<S, R, __VA_ARGS__>::BYTES, &match_shape<S>,                            \
     &launch_fwd<S, CELL, R, MODE, __VA_ARGS__>, &prepare_fwd<S, CELL, R, MODE, __VA_ARGS__>, 0}
// contracted chain (tts::Merge01) of the three-core shape S3: registered under S3, reads S3's blob
#define TTS_FWD_M01(S3, CELL, R, MODE, ...)                                                                \
    {#S3 "(m01)", CELL, MODE, R, tts::FwdSmem<tts::Merge01<S3>, R, __VA_ARGS__>::BYTES, &match_shape<S3>,    \
     &launch_fwd<tts::Merge01<S3>, CELL, R, MODE, __VA_ARGS__>, &prepare_fwd<tts::Merge01<S3>, CELL, R, MODE, __VA_ARGS__>, 1}

// Tune<FTMr, FTI, FSK, TM1, TN1, TM2, TN2, TM3, TN3>: final-stage tile (rows, first-mode slices, k-split)
// and (rows, columns) of the thread tile of stages 1..3
using tts::Tune;
#define TTS_FWD2(S, CELL, R, MODE, ...)                                                                    \
    {#S "(2 CTAs/SM)", CELL, MODE, R, tts::FwdSmem<S, R, __VA_ARGS__>::BYTES, &match_shape<S>,                \
     &launch_fwd<S, CELL, R, MODE, __VA_ARGS__, 2>, &prepare_fwd<S, CELL, R, MODE, __VA_ARGS__, 2>, 0}
// d3 r8 chain with cores 0 and 1 contracted (J = [32, 8], I = [64, 16], RK = [1, 8, 1]): the final stage contracts
// K = 256; two first-mode slices per thread with k split in halves (FTI = FSK = 2): per k-step R + 8 LDS.128 feed 16 R
// FFMA2.  Four slices / four k-splits measured within 0.1 % of it on cfg3 (B200) and need three times the exchange
// space of the reduce-scatter, so the smaller tile stays.
using TU_m01_R2 = Tune<1, 2, 2, 2, 8>;
using TU_m01_R5 = Tune<1, 2, 2, 1, 8>;
const TtsRnnFwdEntry kFwd[] = {
    TTS_FWD(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 1, tts::MODE_RANK1, Tune<1, 2, 2, 1, 8>),
    TTS_FWD(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 1, tts::MODE_XG, Tune<1, 2, 2, 1, 8>),
    TTS_FWD(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 2, tts::MODE_RANK1, Tune<1, 2, 2, 1, 8>),
    TTS_FWD(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 4, tts::MODE_RANK1, Tune<1, 2, 2, 1, 8>),
    TTS_FWD(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 2, tts::MODE_XG, Tune<1, 2, 2, 1, 8>),
    TTS_FWD(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 4, tts::MODE_XG, Tune<1, 2, 2, 1, 8>),
    TTS_FWD(HH_H256_d2r4_gru, TTRNN_CELL_GRU, 1, tts::MODE_RANK1, Tune<1, 2, 2, 1, 8>),
    TTS_FWD(HH_H256_d2r4_gru, TTRNN_CELL_GRU, 2, tts::MODE_RANK1, Tune<1, 2, 2, 1, 8>),
    TTS_FWD2(HH_H256_d2r4_gru, TTRNN_CELL_GRU, 4, tts::MODE_RANK1, Tune<1, 2, 2, 1, 8>),
    TTS_FWD(HH_H256_d2r4_gru, TTRNN_CELL_GRU, 7, tts::MODE_RANK1, Tune<1, 2, 2, 1, 8>),
    TTS_FWD(HH_H256_d2r4_gru, TTRNN_CELL_GRU, 4, tts::MODE_XG, Tune<1, 2, 2, 1, 8>),
    TTS_FWD(HH_H256_d2r4_gru, TTRNN_CELL_GRU, 7, tts::MODE_XG, Tune<1, 2, 2, 1, 8>),
    // one row per CTA: batches that cannot fill the SMs at two rows per CTA (strong scaling: 80 rows per GPU at 8 GPUs)
    TTS_FWD(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 1, tts::MODE_XG, Tune<1, 1, 1, 2, 8, 2, 8>),
    TTS_FWD(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 2, tts::MODE_XG, Tune<1, 1, 1, 2, 8, 2, 8>),
    // three / four rows per CTA: 296 < B <= 592 (the 320 rows per GPU of the 2-GPU strong-scaling point) would otherwise run
    // 64 five-row CTAs on 148 SMs
    TTS_FWD(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 3, tts::MODE_XG, Tune<1, 1, 1, 1, 8, 1, 8>),
    TTS_FWD(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 4, tts::MODE_XG, Tune<1, 1, 1, 1, 8, 1, 8>),
    TTS_FWD(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 5, tts::MODE_XG, Tune<1, 1, 1, 1, 8, 1, 8>),
    TTS_FWD_M01(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 1, tts::MODE_XG, TU_m01_R2),
    TTS_FWD_M01(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 2, tts::MODE_XG, TU_m01_R2),
    TTS_FWD_M01(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 3, tts::MODE_XG, TU_m01_R5),
    TTS_FWD_M01(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 4, tts::MODE_XG, TU_m01_R5),
    TTS_FWD_M01(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 5, tts::MODE_XG, TU_m01_R5),
    TTS_FWD(HH_H768_d2r4_lstm, TTRNN_CELL_LSTM, 2, tts::MODE_XG, Tune<1, 3, 1, 1, 8>),
    TTS_FWD(HH_H768_d2r4_lstm, TTRNN_CELL_LSTM, 4, tts::MODE_XG, Tune<1, 3, 1, 1, 8>),
    TTS_FWD(HH_H256_d4r16_lstm, TTRNN_CELL_LSTM, 1, tts::MODE_XG, Tune<4, 1, 4, 8, 8, 8, 8, 4, 8>),
    TTS_FWD(HH_H1024_d4r8_lstm, TTRNN_CELL_LSTM, 1, tts::MODE_XG, Tune<8, 1, 2, 8, 8, 4, 8, 4, 8>),
};


template <class S, int CELL, int R, int MODE, class TB, bool DWI, int SV = 0, int MINB = 1>
int launch_bwd(const tts::RnnBwdSArgs *a, int grid, cudaStream_t st) {
    tts::k_rnn_bwd_s<S, CELL, R, MODE, TB, DWI, SV, MINB><<<grid, tts::NTHR, tts::BwdSmem<S, R, TB, DWI, SV>::BYTES, st>>>(*a);
    return (int)cudaGetLastError();
}
template <class S, int CELL, int R, int MODE, class TB, bool DWI, int SV = 0, int MINB = 1>
int prepare_bwd(int *occ) {
    auto k = tts::k_rnn_bwd_s<S, CELL, R, MODE, TB, DWI, SV, MINB>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tts::BwdSmem<S, R, TB, DWI, SV>::BYTES);
    if (e != cudaSuccess) return (int)e;
    return (int)cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, k, tts::NTHR, tts::BwdSmem<S, R, TB, DWI, SV>::BYTES);
}
template <class S>
constexpr long long slot_floats() { return tts::blob_floats<S>() + 3LL * S::G * tts::n_in<S>(); }

#define TTS_BWD(S, CELL, R, MODE, ...)                                                                      \
    {#S, CELL, MODE, R, 0, 0, tts::BwdSmem<S, R, __VA_ARGS__, true>::BYTES, slot_floats<S>(), &match_shape<S>, \
     &launch_bwd<S, CELL, R, MODE, __VA_ARGS__, true>, &prepare_bwd<S, CELL, R, MODE, __VA_ARGS__, true>, 0}
#define TTS_BWD_SAVEU(S, CELL, R, MODE, ...)                                                                \
    {#S "(kept u)", CELL, MODE, R, 0, 2, tts::BwdSmem<S, R, __VA_ARGS__, true, 2>::BYTES, slot_floats<S>(),  \
     &match_shape<S>, &launch_bwd<S, CELL, R, MODE, __VA_ARGS__, true, 2>,                                   \
     &prepare_bwd<S, CELL, R, MODE, __VA_ARGS__, true, 2>, 0}
#define TTS_BWD_SPLIT(S, CELL, R, MODE, ...)                                                                \
    {#S "(split)", CELL, MODE, R, 1, 0, tts::BwdSmem<S, R, __VA_ARGS__, false>::BYTES, slot_floats<S>(),     \
     &match_shape<S>, &launch_bwd<S, CELL, R, MODE, __VA_ARGS__, false>,                                     \
     &prepare_bwd<S, CELL, R, MODE, __VA_ARGS__, false>, 0}

// kept gates + split: gate gradients and the dX chain only (no recompute, no in-kernel core gradients)
#define TTS_BWD_SPLIT_SAVEU(S, CELL, R, MODE, ...)                                                          \
    {#S "(split, kept u)", CELL, MODE, R, 1, 2, tts::BwdSmem<S, R, __VA_ARGS__, false, 2>::BYTES, slot_floats<S>(), \
     &match_shape<S>, &launch_bwd<S, CELL, R, MODE, __VA_ARGS__, false, 2>,                                  \
     &prepare_bwd<S, CELL, R, MODE, __VA_ARGS__, false, 2>, 0}

// contracted d3 r8 chain (tts::Merge01), dX-only with kept gates: registered under S3; the gradient slot keeps the
// layout of S3's blob (only the bias gradients are written: the hh core gradients come from the dense accumulation)
#define TTS_BWD_SPLIT_SAVEU_M01(S3, CELL, R, MODE, ...)                                                     \
    {#S3 "(m01, split, kept u)", CELL, MODE, R, 1, 2, tts::BwdSmem<tts::Merge01<S3>, R, __VA_ARGS__, false, 2>::BYTES, \
     slot_floats<S3>(), &match_shape<S3>, &launch_bwd<tts::Merge01<S3>, CELL, R, MODE, __VA_ARGS__, false, 2>,    \
     &prepare_bwd<tts::Merge01<S3>, CELL, R, MODE, __VA_ARGS__, false, 2>, 1}

// the same with the register budget of two co-resident CTAs per SM (one-row variants: 80 KB of shared memory each).
// Measured dead end (round 2, cfg3 shape, 196 / 296 rows): two co-resident one-row CTAs take 2.61 ms per layer-pass
// against 2.33 ms for one two-row CTA per SM -- the per-step latency chain does not overlap across CTAs.  Not registered.
#define TTS_BWD_SPLIT_SAVEU2(S, CELL, R, MODE, ...)                                                         \
    {#S "(split, kept u, 2 CTAs/SM)", CELL, MODE, R, 1, 2, tts::BwdSmem<S, R, __VA_ARGS__, false, 2>::BYTES, slot_floats<S>(), \
     &match_shape<S>, &launch_bwd<S, CELL, R, MODE, __VA_ARGS__, false, 2, 2>,                               \
     &prepare_bwd<S, CELL, R, MODE, __VA_ARGS__, false, 2, 2>, 0}

// TuneB<forward Tune, BTM0..3 (rows per thread of bwd-data stage k), BSP (split of the last bwd-data
// stage), WTK0..3 (kappa rows of the register tile of bwd-weight stage k)>
using tts::TuneB;
using TB_d2 = TuneB<Tune<1, 2, 2, 1, 8>, 1, 1, 1, 1, 8, 8, 8, 8, 8>;
using TB_d3_R5 = TuneB<Tune<1, 1, 1, 1, 8, 1, 8>, 1, 1, 1, 1, 8, 4, 8, 4, 4>;
using TB_d3_R2 = TuneB<Tune<1, 1, 1, 2, 8, 2, 8>, 1, 1, 1, 1, 8, 4, 8, 4, 4>;
// cfg5: split backward (recurrent kernel propagates dh/dc only); last bwd-data stage split 4 ways
using TB_h1024_split = TuneB<Tune<8, 1, 2, 8, 8, 4, 8, 4, 8>, 8, 4, 4, 2, 4, 4, 4, 4, 4>;
using TB_d3_R3 = TuneB<Tune<1, 1, 1, 1, 8, 1, 8>, 1, 1, 1, 1, 8, 4, 8, 4, 4>;
// dX-only kernels of the d3r8 chain: no core-gradient registers, so two rows per thread in the bwd-data stages
using TB_d3_split_R2 = TuneB<Tune<1, 1, 1, 2, 8, 2, 8>, 2, 2, 1, 1, 8, 4, 8, 4, 4>;
using TB_d3_split_R3 = TuneB<Tune<1, 1, 1, 1, 8, 1, 8>, 2, 2, 1, 1, 8, 4, 8, 4, 4>;
// d4 r16 (cfg4 shape) training: dX-only kernel with kept gates; last bwd-data stage split 4 ways
// H = 768 d2 r4: dX-only kernel with kept gates (the fused variant's core-gradient tiles do not divide 256 threads)
using TB_h768_split = TuneB<Tune<1, 3, 1, 1, 8>, 1, 1, 1, 1, 2, 8, 8, 8, 8>;
using TB_d4r16_split = TuneB<Tune<4, 1, 4, 8, 8, 8, 8, 4, 8>, 8, 8, 4, 1, 4, 4, 4, 4, 4>;
// contracted d3 r8 chain, dX only: bwd-data stage 0 (K = 256, 64 gate rows) two rows per thread, stage 1 as stage 2 of
// the three-core chain (split 8 ways); the forward tile only sets the ownership of hidden units (one per thread)
using TB_m01_split = TuneB<Tune<1, 1, 1, 1, 8>, 2, 1, 1, 1, 8, 4, 8, 4, 4>;
const TtsRnnBwdEntry kBwd[] = {
    TTS_BWD(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 2, tts::MODE_RANK1, TB_d2),
    TTS_BWD(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 4, tts::MODE_RANK1, TB_d2),
    TTS_BWD(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 2, tts::MODE_XG, TB_d2),
    TTS_BWD(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 4, tts::MODE_XG, TB_d2),
    TTS_BWD(HH_H256_d2r4_gru, TTRNN_CELL_GRU, 4, tts::MODE_RANK1, TB_d2),
    TTS_BWD(HH_H256_d2r4_gru, TTRNN_CELL_GRU, 7, tts::MODE_RANK1, TB_d2),
    TTS_BWD(HH_H256_d2r4_gru, TTRNN_CELL_GRU, 4, tts::MODE_XG, TB_d2),
    TTS_BWD(HH_H256_d2r4_gru, TTRNN_CELL_GRU, 7, tts::MODE_XG, TB_d2),
    TTS_BWD_SAVEU(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 1, tts::MODE_RANK1, TB_d2),
    TTS_BWD_SAVEU(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 1, tts::MODE_XG, TB_d2),
    TTS_BWD_SAVEU(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 2, tts::MODE_RANK1, TB_d2),
    TTS_BWD_SAVEU(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 4, tts::MODE_RANK1, TB_d2),
    TTS_BWD_SAVEU(HH_H256_d2r4_gru, TTRNN_CELL_GRU, 1, tts::MODE_RANK1, TB_d2),
    TTS_BWD_SAVEU(HH_H256_d2r4_gru, TTRNN_CELL_GRU, 2, tts::MODE_RANK1, TB_d2),
    TTS_BWD_SAVEU(HH_H256_d2r4_gru, TTRNN_CELL_GRU, 4, tts::MODE_RANK1, TB_d2),
    TTS_BWD_SAVEU(HH_H256_d2r4_gru, TTRNN_CELL_GRU, 7, tts::MODE_RANK1, TB_d2),
    TTS_BWD_SAVEU(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 2, tts::MODE_XG, TB_d2),
    TTS_BWD_SAVEU(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 4, tts::MODE_XG, TB_d2),
    TTS_BWD_SAVEU(HH_H256_d2r4_gru, TTRNN_CELL_GRU, 4, tts::MODE_XG, TB_d2),
    TTS_BWD_SAVEU(HH_H256_d2r4_gru, TTRNN_CELL_GRU, 7, tts::MODE_XG, TB_d2),
    TTS_BWD_SAVEU(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 2, tts::MODE_XG, TB_d3_R2),
    TTS_BWD_SAVEU(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 3, tts::MODE_XG, TB_d3_R3),
    TTS_BWD(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 2, tts::MODE_XG, TB_d3_R2),
    TTS_BWD(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 3, tts::MODE_XG, TB_d3_R3),
    TTS_BWD_SPLIT(HH_H1024_d4r8_lstm, TTRNN_CELL_LSTM, 1, tts::MODE_XG, TB_h1024_split),
    TTS_BWD_SPLIT_SAVEU(HH_H256_d4r16_lstm, TTRNN_CELL_LSTM, 1, tts::MODE_XG, TB_d4r16_split),
    TTS_BWD_SPLIT_SAVEU(HH_H768_d2r4_lstm, TTRNN_CELL_LSTM, 2, tts::MODE_XG, TB_h768_split),
    TTS_BWD_SPLIT_SAVEU(HH_H768_d2r4_lstm, TTRNN_CELL_LSTM, 3, tts::MODE_XG, TB_h768_split),
    // d2 r4 chains with a rank-one input (cfg1 / cfg2): dX-only kernels that write delta_hh, hh core gradients on the
    // tensor cores (dW_hh^T = H_prev^T delta), ih / bias gradients still accumulated in registers
    TTS_BWD_SPLIT_SAVEU(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 1, tts::MODE_RANK1, TB_d2),
    TTS_BWD_SPLIT_SAVEU(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 2, tts::MODE_RANK1, TB_d2),
    TTS_BWD_SPLIT_SAVEU(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 4, tts::MODE_RANK1, TB_d2),
    TTS_BWD_SPLIT_SAVEU(HH_H256_d2r4_gru, TTRNN_CELL_GRU, 2, tts::MODE_RANK1, TB_d2),
    TTS_BWD_SPLIT_SAVEU(HH_H256_d2r4_gru, TTRNN_CELL_GRU, 4, tts::MODE_RANK1, TB_d2),
    TTS_BWD_SPLIT_SAVEU(HH_H256_d2r4_gru, TTRNN_CELL_GRU, 7, tts::MODE_RANK1, TB_d2),
    // d2 r4 chain behind a projected input (the rank-padded params_model.py default, cfg3-alt): dX-only kernels, core
    // gradients on the tensor cores
    TTS_BWD_SPLIT_SAVEU(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 1, tts::MODE_XG, TB_d2),
    TTS_BWD_SPLIT_SAVEU(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 2, tts::MODE_XG, TB_d2),
    TTS_BWD_SPLIT_SAVEU(HH_H256_d2r4_lstm, TTRNN_CELL_LSTM, 4, tts::MODE_XG, TB_d2),
    TTS_BWD_SPLIT_SAVEU(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 1, tts::MODE_XG, TB_d3_split_R2),
    TTS_BWD_SPLIT_SAVEU(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 2, tts::MODE_XG, TB_d3_split_R2),
    TTS_BWD_SPLIT_SAVEU(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 3, tts::MODE_XG, TB_d3_split_R3),
    // four rows fit once the contracted chain drops the second X_k slot (209 KB; 246 KB for the three-core chain)
    TTS_BWD_SPLIT_SAVEU_M01(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 1, tts::MODE_XG, TB_m01_split),
    TTS_BWD_SPLIT_SAVEU_M01(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 2, tts::MODE_XG, TB_m01_split),
    TTS_BWD_SPLIT_SAVEU_M01(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 3, tts::MODE_XG, TB_m01_split),
    TTS_BWD_SPLIT_SAVEU_M01(HH_H256_d3r8_lstm, TTRNN_CELL_LSTM, 4, tts::MODE_XG, TB_m01_split),
};


// ---- batched TT matvec ---------------------------------------------------------------------------
template <class S, int R, class TU>
int launch_tf(const tts::TtlFwdSArgs *a, int grid, cudaStream_t st) {
    tts::k_ttlin_fwd_s<S, R, TU><<<grid, tts::NTHR, tts::TtlFwdSmem<S, R, TU>::BYTES, st>>>(*a);
    return (int)cudaGetLastError();
}
template <class S, int R, class TU>
int prepare_tf(int *occ) {
    auto k = tts::k_ttlin_fwd_s<S, R, TU>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tts::TtlFwdSmem<S, R, TU>::BYTES);
    if (e != cudaSuccess) return (int)e;
    return (int)cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, k, tts::NTHR, tts::TtlFwdSmem<S, R, TU>::BYTES);
}
template <class S, int R, class TB, bool DX>
int launch_tb(const tts::TtlBwdSArgs *a, int grid, cudaStream_t st) {
    tts::k_ttlin_bwd_s<S, R, TB, DX><<<grid, tts::NTHR, tts::TtlBwdSmem<S, R, TB, DX>::BYTES, st>>>(*a);
    return (int)cudaGetLastError();
}
template <class S, int R, class TB, bool DX>
int prepare_tb(int *occ) {
    auto k = tts::k_ttlin_bwd_s<S, R, TB, DX>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tts::TtlBwdSmem<S, R, TB, DX>::BYTES);
    if (e != cudaSuccess) return (int)e;
    return (int)cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, k, tts::NTHR, tts::TtlBwdSmem<S, R, TB, DX>::BYTES);
}
#define TTS_TF(S, R, ...) \
    {#S, R, tts::TtlFwdSmem<S, R, __VA_ARGS__>::BYTES, &match_shape<S>, &launch_tf<S, R, __VA_ARGS__>, &prepare_tf<S, R, __VA_ARGS__>}
#define TTS_TB(S, R, DX, ...) \
    {#S, R, DX, tts::TtlBwdSmem<S, R, __VA_ARGS__, DX>::BYTES, &match_shape<S>, &launch_tb<S, R, __VA_ARGS__, DX>, &prepare_tb<S, R, __VA_ARGS__, DX>}

using TU_ih40_d3 = Tune<1, 1, 1, 1, 8, 1, 4>;
using TU_ih256_d3 = Tune<1, 1, 1, 1, 8, 1, 8>;
using TU_ih256_d3_R4 = Tune<1, 1, 1, 2, 8, 2, 8>;
using TU_ih256_d4r8 = Tune<2, 1, 1, 8, 8, 4, 8, 2, 8>;
using TU_ih40_d4r16 = Tune<1, 1, 1, 4, 8, 2, 8, 1, 4>;
using TU_ih256_d4r16 = Tune<1, 1, 1, 8, 8, 8, 8, 4, 8>;
const TtsTtlFwdEntry kTtlFwd[] = {
    TTS_TF(IH_40_H256_d3r8, 8, TU_ih40_d3),
    TTS_TF(IH_256_H256_d3r8, 4, TU_ih256_d3_R4),
    TTS_TF(IH_256_H1024_d4r8, 1, TU_ih256_d4r8),
    TTS_TF(IH_40_H256_d4r16, 2, TU_ih40_d4r16),
    TTS_TF(IH_256_H256_d4r16, 1, TU_ih256_d4r16),
};
using TBI_ih40_d3 = TuneB<TU_ih40_d3, 1, 1, 1, 1, 8, 4, 8, 8, 4>;
using TBI_ih256_d3 = TuneB<TU_ih256_d3, 1, 1, 1, 1, 8, 4, 8, 4, 4>;
using TBI_hhw_h1024 = TuneB<Tune<1, 1, 1, 8, 8, 4, 8, 4, 8>, 8, 4, 4, 1, 4, 4, 4, 8, 4>;
using TBI_ih256_d4r8 = TuneB<TU_ih256_d4r8, 8, 4, 2, 1, 4, 4, 8, 8, 4>;
const TtsTtlBwdEntry kTtlBwd[] = {
    TTS_TB(IH_40_H256_d3r8, 4, false, TBI_ih40_d3),
    TTS_TB(IH_256_H256_d3r8, 3, true, TBI_ih256_d3),
    // without dX: the H-row projection of the dense dW^T onto the cores (once per layer and call; same shape for ih and hh)
    TTS_TB(IH_256_H256_d3r8, 3, false, TBI_ih256_d3),
    TTS_TB(IH_256_H1024_d4r8, 1, false, TBI_ih256_d4r8),
    TTS_TB(HHW_H1024_d4r8, 1, false, TBI_hhw_h1024),
};

}  // namespace

// text table of every registered static kernel: "kind name R smem_bytes fits\n" (tests assert that all fit)
int tts_dump_entries(char *buf, int cap) {
    int n = 0;
    auto put = [&](const char *kind, const char *name, int R, size_t smem) {
        if (n < cap) n += snprintf(buf + n, cap - n, "%s|%s|%d|%zu|%d\n", kind, name, R, smem, smem <= kMaxSmem ? 1 : 0);
    };
    for (const auto &e : kFwd) put("rnn_fwd", e.name, e.R, e.smem);
    for (const auto &e : kBwd) put("rnn_bwd", e.name, e.R, e.smem);
    for (const auto &e : kTtlFwd) put("ttl_fwd", e.name, e.R, e.smem);
    for (const auto &e : kTtlBwd) put("ttl_bwd", e.name, e.R, e.smem);
    return n;
}

const TtsTtlFwdEntry *tts_find_ttl_fwd(const ttrnn_tt_shape *s, long long rows) {
    if (rows < 64) return nullptr;                  // tiny calls (rank-one helper rows) stay on the generic kernel
    for (const auto &e : kTtlFwd)
        if (e.match(s) && e.smem <= kMaxSmem) return &e;
    return nullptr;
}
const TtsTtlBwdEntry *tts_find_ttl_bwd(const ttrnn_tt_shape *s, long long rows, int want_dx) {
    if (rows < 64) return nullptr;
    for (const auto &e : kTtlBwd)
        if (e.match(s) && e.smem <= kMaxSmem && e.want_dx == (want_dx ? 1 : 0)) return &e;
    return nullptr;
}

// kept gates (saved == 2): a "split" variant (gate gradients + dX chain only; core gradients by the dense
// accumulation outside) does a third of the work per row of the fused variant and is preferred when the caller
// can run the dense accumulation (split_kept_ok)
// merge != 0: the contracted-chain variants (merged = 1) replace the three-core ones wherever one of them passes `ok`;
// otherwise only the three-core variants compete.  Returns the `merged` value the candidates must have.
template <class E, size_t N, class F>
static int merged_wanted(const E (&tab)[N], int merge, F ok) {
    if (merge)
        for (const auto &e : tab)
            if (e.merged && ok(e)) return 1;
    return 0;
}

static bool use_split_kept(const ttrnn_tt_shape *hh, int cell, int mode, int saved, int split_kept_ok) {
    if (saved != 2 || !split_kept_ok) return false;
    for (const auto &e : kBwd)
        if (e.cell == cell && e.mode == mode && e.saved == 2 && e.split && e.match(hh) && e.smem <= kMaxSmem) return true;
    return false;
}

const TtsRnnBwdEntry *tts_find_rnn_bwd(const ttrnn_tt_shape *hh, int cell, int mode, long long B, int sms, int prefer_R,
                                       int saved, int split_kept_ok, int merge) {
    const TtsRnnBwdEntry *best = nullptr;
    const bool only_split = use_split_kept(hh, cell, mode, saved, split_kept_ok);
    auto ok = [&](const TtsRnnBwdEntry &e) {
        return e.cell == cell && e.mode == mode && e.saved == saved && e.match(hh) && e.smem <= kMaxSmem &&
               (saved != 2 || (e.split != 0) == only_split);
    };
    const int mw = merged_wanted(kBwd, merge, ok);
    if (prefer_R > 0)
        for (const auto &e : kBwd)
            if (ok(e) && e.merged == mw && e.R == prefer_R) return &e;
    long long best_cost = 0;
    for (const auto &e : kBwd) {
        if (!ok(e) || e.merged != mw) continue;
        const long long tiles = (B + e.R - 1) / e.R;
        const long long waves = (tiles + sms - 1) / sms;
        const long long cost = waves * (2 * e.R + 3);
        if (!best || cost < best_cost || (cost == best_cost && e.R > best->R)) {
            best = &e;
            best_cost = cost;
        }
    }
    return best;
}

int tts_plan_rnn_bwd(const ttrnn_tt_shape *hh, int cell, int mode, long long B, int sms, int prefer_R, int saved,
                     int split_kept_ok, int merge, const TtsRnnBwdEntry *entry[2], long long row0[2], long long rows[2]) {
    entry[0] = entry[1] = nullptr;
    row0[0] = row0[1] = rows[0] = rows[1] = 0;
    if (prefer_R > 0) {
        entry[0] = tts_find_rnn_bwd(hh, cell, mode, B, sms, prefer_R, saved, split_kept_ok, merge);
        rows[0] = B;
        return entry[0] ? 1 : 0;
    }
    const bool only_split = use_split_kept(hh, cell, mode, saved, split_kept_ok);
    auto ok0 = [&](const TtsRnnBwdEntry &e) {
        return e.cell == cell && e.mode == mode && e.saved == saved && e.match(hh) && e.smem <= kMaxSmem &&
               (saved != 2 || (e.split != 0) == only_split);
    };
    const int mw = merged_wanted(kBwd, merge, ok0);
    auto ok = [&](const TtsRnnBwdEntry &e) { return ok0(e) && e.merged == mw; };
    // cost of a wave of R rows per CTA ~ (1 + R): one unit of per-step overhead (barriers, gate phase) per row of work
    auto wave_cost = [&](const TtsRnnBwdEntry &e, long long nrows) {
        const long long tiles = (nrows + e.R - 1) / e.R;
        return ((tiles + sms - 1) / sms) * (1 + e.R);
    };
    long long best = 0;
    int n = 0;
    for (const auto &a : kBwd) {
        if (!ok(a)) continue;
        const long long c1 = wave_cost(a, B);
        if (n == 0 || c1 < best || (c1 == best && n == 1 && a.R > entry[0]->R)) {
            best = c1; n = 1;
            entry[0] = &a; entry[1] = nullptr;
            row0[0] = 0; rows[0] = B; rows[1] = 0;
        }
        const long long full = B / ((long long)a.R * sms);           // whole waves of variant a
        const long long rem = B - full * a.R * sms;
        if (full < 1 || rem == 0) continue;
        for (const auto &b : kBwd) {
            if (!ok(b) || b.split != a.split) continue;
            const long long c2 = full * (1 + a.R) + wave_cost(b, rem);
            if (c2 < best) {
                best = c2; n = 2;
                entry[0] = &a; entry[1] = &b;
                row0[0] = 0; rows[0] = full * a.R * sms;
                row0[1] = rows[0]; rows[1] = rem;
            }
        }
    }
    return n;
}

const TtsRnnFwdEntry *tts_find_rnn_fwd(const ttrnn_tt_shape *hh, int cell, int mode, long long B, int sms, int prefer_R,
                                       int merge) {
    const TtsRnnFwdEntry *best = nullptr;
    auto ok = [&](const TtsRnnFwdEntry &e) { return e.cell == cell && e.mode == mode && e.match(hh) && e.smem <= kMaxSmem; };
    const int mw = merged_wanted(kFwd, merge, ok);
    if (prefer_R > 0)
        for (const auto &e : kFwd)
            if (ok(e) && e.merged == mw && e.R == prefer_R) return &e;
    long long best_cost = 0;
    for (const auto &e : kFwd) {
        if (!ok(e) || e.merged != mw) continue;
        const long long tiles = (B + e.R - 1) / e.R;
        const long long waves = (tiles + sms - 1) / sms;
        // time of a wave of R rows per CTA ~ (1.5 + R): a latency floor per step (barriers, shared-memory round trips) plus
        // the per-row work; without the floor a batch of 320 would run as three waves of one-row CTAs
        const long long cost = waves * (2 * e.R + 3);
        if (!best || cost < best_cost || (cost == best_cost && e.R > best->R)) {
            best = &e;
            best_cost = cost;
        }
    }
    return best;
}
