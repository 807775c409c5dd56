// Host-side registry of the statically specialised kernels (tt_static.cuh / tt_static_inst.cu).
#pragma once
#include <cuda_runtime.h>
#include "../../include/ttrnn_b200.h"

namespace tts {
struct RnnFwdSArgs;
struct RnnBwdSArgs;
struct TtlFwdSArgs;
struct TtlBwdSArgs;
}

struct TtsRnnFwdEntry {
    const char *name;
    int cell, mode, R;
    size_t smem;
    bool (*match)(const ttrnn_tt_shape *hh);
    int (*launch)(const tts::RnnFwdSArgs *args, int grid, cudaStream_t st);   // 0 = ok, else cudaError_t
    int (*prepare)(int *max_blocks_per_sm);                                  // sets attributes; 0 = ok
    int merged;                                                               // 1: runs the chain with cores 0 and 1 contracted
};

// best registered forward kernel for (hh shape, cell, mode) at batch B on `sms` SMs, or nullptr.  merge != 0: where a
// contracted-chain variant (tts::Merge01) serves the query, only those compete; merge == 0: they are never chosen.
const TtsRnnFwdEntry *tts_find_rnn_fwd(const ttrnn_tt_shape *hh, int cell, int mode, long long B, int sms,
                                       int prefer_R, int merge);

struct TtsRnnBwdEntry {
    const char *name;
    int cell, mode, R;
    int split;                                                               // 1: core gradients come from a batched kernel
    int saved;                                                               // 2: consumes the gate activations kept by the forward, 0: recomputes
    size_t smem;
    long long slot_floats;                                                   // floats per gradient slot
    bool (*match)(const ttrnn_tt_shape *hh);
    int (*launch)(const tts::RnnBwdSArgs *args, int grid, cudaStream_t st);
    int (*prepare)(int *max_blocks_per_sm);
    int merged;                                                               // 1: contracted chain (dX only; gradient slot of the 3-core blob)
};
// split_kept_ok: with saved == 2, prefer the split variants (gate gradients + dX chain only) when registered;
// the caller then accumulates the hh core gradients in the dense order.  merge: as for tts_find_rnn_fwd
const TtsRnnBwdEntry *tts_find_rnn_bwd(const ttrnn_tt_shape *hh, int cell, int mode, long long B, int sms,
                                       int prefer_R, int saved, int split_kept_ok, int merge);

// Row plan of one BPTT launch: up to two phases (kernel variant, first row, row count).  When the batch does
// not fill whole waves of the best variant, the tail runs on a variant with fewer rows per CTA instead of
// a mostly idle second wave (cfg3: 640 rows = one wave of 148 x 3 rows + one wave of 98 x 2 rows).
// Returns the number of phases (0 = no registered kernel).
int tts_plan_rnn_bwd(const ttrnn_tt_shape *hh, int cell, int mode, long long B, int sms, int prefer_R, int saved,
                     int split_kept_ok, int merge, const TtsRnnBwdEntry *entry[2], long long row0[2], long long rows[2]);

struct TtsTtlFwdEntry {
    const char *name;
    int R;
    size_t smem;
    bool (*match)(const ttrnn_tt_shape *s);
    int (*launch)(const tts::TtlFwdSArgs *args, int grid, cudaStream_t st);
    int (*prepare)(int *max_blocks_per_sm);
};
struct TtsTtlBwdEntry {
    const char *name;
    int R, want_dx;
    size_t smem;
    bool (*match)(const ttrnn_tt_shape *s);
    int (*launch)(const tts::TtlBwdSArgs *args, int grid, cudaStream_t st);
    int (*prepare)(int *max_blocks_per_sm);
};
const TtsTtlFwdEntry *tts_find_ttl_fwd(const ttrnn_tt_shape *s, long long rows);
const TtsTtlBwdEntry *tts_find_ttl_bwd(const ttrnn_tt_shape *s, long long rows, int want_dx);

// text table of the registry (kind|name|R|smem bytes|fits 227 KB), returns the number of characters written
int tts_dump_entries(char *buf, int cap);
