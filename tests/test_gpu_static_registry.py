"""Every statically specialised kernel of the registry (csrc/tt_static_inst.cu) against the FP64 oracle.

The ledger below holds one case per registry entry, keyed by (kind, name, rows per CTA, cell, input mode, saved gates,
split, merged chain) as ttrnn_static_kernel_keys() prints it; test_static_registry_cpu.py asserts that its keys are
exactly the registry's, so a new TTS_FWD / TTS_BWD / TTS_TF / TTS_TB line needs a case here.  A case is a model and
the options that force the entry (rows per CTA, kept gates, split variants, contracted chain, TT-chain ih route), with
the row plan and row groups off so that one launch covers the whole batch.  Which kernel ran is read from the launch
counters of ttrnn_static_kernel_launches(), not from describe; the recurrent routes must also be the ones describe
names.

Each case runs at three batch sizes: fewer rows than one tile, a ragged last tile within one wave, and more tiles than
CTAs (every static kernel loops `tile_i += gridDim.x`, so a CTA then runs several tiles; the launch records prove it).
Outputs, final states and the input / initial-state gradients are compared separately over the rows of the first round
of tiles and over the later ones, and a second backward with the upstream gradient on later-round rows only checks
the parameter gradients that tiles after a CTA's first make.  Where the route survives time chunks, the large batch
runs chunked as well, and every forward kernel must give bit-identical results under torch.no_grad().

Tolerances: 1e-5 forward, 1e-4 gradients, norm-wise relative.
"""
import ctypes
import io
import re
from collections import namedtuple
from contextlib import contextmanager, redirect_stdout

import pytest
import torch

pytestmark = pytest.mark.gpu

LSTM, GRU, NA = 0, 1, -1          # TTRNN_CELL_*; NA: column does not apply (TT-matvec kernels)
XG, RANK1 = 0, 1                  # input modes (tts::MODE_XG / MODE_RANK1)

D2_LSTM, D2_GRU, D3, H768, D4R16, H1024 = ("HH_H256_d2r4_lstm", "HH_H256_d2r4_gru", "HH_H256_d3r8_lstm",
                                           "HH_H768_d2r4_lstm", "HH_H256_d4r16_lstm", "HH_H1024_d4r8_lstm")


def fwd(name, R, cell, mode, merged=0):
    return ("rnn_fwd", name, R, cell, mode, 0, 0, merged)


def bwd(name, R, cell, mode, saved, split, merged=0):
    return ("rnn_bwd", name, R, cell, mode, saved, split, merged)


def ttl_fwd(name, R):
    return ("ttl_fwd", name, R, NA, NA, NA, 0, 0)


def ttl_bwd(name, R, want_dx):
    return ("ttl_bwd", name, R, NA, NA, NA, 0 if want_dx else 1, 0)


# name suffixes of the registry macros
FUSED, KEPT, SPLIT, SPLIT_KEPT, M01, M01_SPLIT_KEPT, TWO_CTAS = (
    "", "(kept u)", "(split)", "(split, kept u)", "(m01)", "(m01, split, kept u)", "(2 CTAs/SM)")

# options that select a variant (on top of row_plan = 0, row_groups = 0)
RECOMPUTE = {"save_u_bytes": 0}              # no kept gates: the recompute kernels
FUSED_KEPT = {"split_kept": 0}               # kept gates, core gradients inside the BPTT kernel
THREE_CORE = {"merge_cores": 0}              # d3 r8: the three-core chain also for the dX-only kernels
MERGED_FWD = {"merge_cores": 2}              # d3 r8: the contracted chain also for the forward
TT_IH = {"dense_ih": 0}                      # ih projection through the TT chain (the batched TT-matvec kernels)


def rows(f, b):
    return {"static_rows_fwd": f, "static_rows_bwd": b}


# id, (cell, I, H, d, r), options, x.requires_grad, chunked run, targets.  One layer: the entries match on the hh
# shape, and an input of 256 features gives layer 0 the ih shapes of the inner layers.
Case = namedtuple("Case", "id model opts xgrad chunk targets")
CASES = [
    # d2 r4 TT-LSTM, rank-one input (cfg1): split kept-gates kernels need the whole sequence in one chunk
    Case("lstm_rank1_r1_split", ("lstm", 1, 256, 2, 4), rows(1, 1), False, False,
         [fwd(D2_LSTM, 1, LSTM, RANK1), bwd(D2_LSTM + SPLIT_KEPT, 1, LSTM, RANK1, 2, 1)]),
    Case("lstm_rank1_r2_split", ("lstm", 1, 256, 2, 4), rows(2, 2), False, False,
         [fwd(D2_LSTM, 2, LSTM, RANK1), bwd(D2_LSTM + SPLIT_KEPT, 2, LSTM, RANK1, 2, 1)]),
    Case("lstm_rank1_r4_split", ("lstm", 1, 256, 2, 4), rows(4, 4), False, False,
         [fwd(D2_LSTM, 4, LSTM, RANK1), bwd(D2_LSTM + SPLIT_KEPT, 4, LSTM, RANK1, 2, 1)]),
    Case("lstm_rank1_r1_kept", ("lstm", 1, 256, 2, 4), {**rows(2, 1), **FUSED_KEPT}, False, True,
         [bwd(D2_LSTM + KEPT, 1, LSTM, RANK1, 2, 0)]),
    Case("lstm_rank1_r2_kept", ("lstm", 1, 256, 2, 4), {**rows(2, 2), **FUSED_KEPT}, False, True,
         [bwd(D2_LSTM + KEPT, 2, LSTM, RANK1, 2, 0)]),
    Case("lstm_rank1_r4_kept", ("lstm", 1, 256, 2, 4), {**rows(4, 4), **FUSED_KEPT}, False, True,
         [bwd(D2_LSTM + KEPT, 4, LSTM, RANK1, 2, 0)]),
    Case("lstm_rank1_r2_recompute", ("lstm", 1, 256, 2, 4), {**rows(1, 2), **RECOMPUTE}, False, True,
         [bwd(D2_LSTM, 2, LSTM, RANK1, 0, 0)]),
    Case("lstm_rank1_r4_recompute", ("lstm", 1, 256, 2, 4), {**rows(4, 4), **RECOMPUTE}, False, True,
         [bwd(D2_LSTM, 4, LSTM, RANK1, 0, 0)]),
    # d2 r4 TT-LSTM behind a projected input (cfg3-alt)
    Case("lstm_xg_r1_split", ("lstm", 40, 256, 2, 4), rows(1, 1), True, True,
         [fwd(D2_LSTM, 1, LSTM, XG), bwd(D2_LSTM + SPLIT_KEPT, 1, LSTM, XG, 2, 1)]),
    Case("lstm_xg_r2_split", ("lstm", 40, 256, 2, 4), rows(2, 2), True, True,
         [fwd(D2_LSTM, 2, LSTM, XG), bwd(D2_LSTM + SPLIT_KEPT, 2, LSTM, XG, 2, 1)]),
    Case("lstm_xg_r4_split", ("lstm", 40, 256, 2, 4), rows(4, 4), False, True,
         [fwd(D2_LSTM, 4, LSTM, XG), bwd(D2_LSTM + SPLIT_KEPT, 4, LSTM, XG, 2, 1)]),
    Case("lstm_xg_r1_kept", ("lstm", 40, 256, 2, 4), {**rows(1, 1), **FUSED_KEPT}, True, True,
         [bwd(D2_LSTM + KEPT, 1, LSTM, XG, 2, 0)]),
    Case("lstm_xg_r2_kept", ("lstm", 40, 256, 2, 4), {**rows(2, 2), **FUSED_KEPT}, False, True,
         [bwd(D2_LSTM + KEPT, 2, LSTM, XG, 2, 0)]),
    Case("lstm_xg_r4_kept", ("lstm", 40, 256, 2, 4), {**rows(4, 4), **FUSED_KEPT}, True, True,
         [bwd(D2_LSTM + KEPT, 4, LSTM, XG, 2, 0)]),
    Case("lstm_xg_r2_recompute", ("lstm", 40, 256, 2, 4), {**rows(2, 2), **RECOMPUTE}, True, True,
         [bwd(D2_LSTM, 2, LSTM, XG, 0, 0)]),
    Case("lstm_xg_r4_recompute", ("lstm", 40, 256, 2, 4), {**rows(4, 4), **RECOMPUTE}, False, True,
         [bwd(D2_LSTM, 4, LSTM, XG, 0, 0)]),
    # d2 r4 TT-GRU, rank-one input (cfg2)
    Case("gru_rank1_r1_kept", ("gru", 1, 256, 2, 4), {**rows(1, 1), **FUSED_KEPT}, False, True,
         [fwd(D2_GRU, 1, GRU, RANK1), bwd(D2_GRU + KEPT, 1, GRU, RANK1, 2, 0)]),
    Case("gru_rank1_r2_split", ("gru", 1, 256, 2, 4), rows(2, 2), False, False,
         [fwd(D2_GRU, 2, GRU, RANK1), bwd(D2_GRU + SPLIT_KEPT, 2, GRU, RANK1, 2, 1)]),
    Case("gru_rank1_r4_split", ("gru", 1, 256, 2, 4), rows(4, 4), False, False,
         [fwd(D2_GRU + TWO_CTAS, 4, GRU, RANK1), bwd(D2_GRU + SPLIT_KEPT, 4, GRU, RANK1, 2, 1)]),
    Case("gru_rank1_r7_split", ("gru", 1, 256, 2, 4), rows(7, 7), False, False,
         [fwd(D2_GRU, 7, GRU, RANK1), bwd(D2_GRU + SPLIT_KEPT, 7, GRU, RANK1, 2, 1)]),
    Case("gru_rank1_r2_kept", ("gru", 1, 256, 2, 4), {**rows(2, 2), **FUSED_KEPT}, False, True,
         [bwd(D2_GRU + KEPT, 2, GRU, RANK1, 2, 0)]),
    Case("gru_rank1_r4_kept", ("gru", 1, 256, 2, 4), {**rows(4, 4), **FUSED_KEPT}, False, True,
         [bwd(D2_GRU + KEPT, 4, GRU, RANK1, 2, 0)]),
    Case("gru_rank1_r7_kept", ("gru", 1, 256, 2, 4), {**rows(7, 7), **FUSED_KEPT}, False, True,
         [bwd(D2_GRU + KEPT, 7, GRU, RANK1, 2, 0)]),
    Case("gru_rank1_r4_recompute", ("gru", 1, 256, 2, 4), {**rows(4, 4), **RECOMPUTE}, False, True,
         [bwd(D2_GRU, 4, GRU, RANK1, 0, 0)]),
    Case("gru_rank1_r7_recompute", ("gru", 1, 256, 2, 4), {**rows(7, 7), **RECOMPUTE}, False, True,
         [bwd(D2_GRU, 7, GRU, RANK1, 0, 0)]),
    # d2 r4 TT-GRU behind a projected input: no split variant, kept gates go to the fused kernels
    Case("gru_xg_r4_kept", ("gru", 40, 256, 2, 4), rows(4, 4), True, True,
         [fwd(D2_GRU, 4, GRU, XG), bwd(D2_GRU + KEPT, 4, GRU, XG, 2, 0)]),
    Case("gru_xg_r7_kept", ("gru", 40, 256, 2, 4), rows(7, 7), False, True,
         [fwd(D2_GRU, 7, GRU, XG), bwd(D2_GRU + KEPT, 7, GRU, XG, 2, 0)]),
    Case("gru_xg_r4_recompute", ("gru", 40, 256, 2, 4), {**rows(4, 4), **RECOMPUTE}, False, True,
         [bwd(D2_GRU, 4, GRU, XG, 0, 0)]),
    Case("gru_xg_r7_recompute", ("gru", 40, 256, 2, 4), {**rows(7, 7), **RECOMPUTE}, True, True,
         [bwd(D2_GRU, 7, GRU, XG, 0, 0)]),
    # d3 r8 TT-LSTM (cfg3): three-core and contracted (m01) chains
    Case("d3_r1_m01_split", ("lstm", 40, 256, 3, 8), rows(1, 1), True, True,
         [fwd(D3, 1, LSTM, XG), bwd(D3 + M01_SPLIT_KEPT, 1, LSTM, XG, 2, 1, 1)]),
    Case("d3_r2_m01_split", ("lstm", 40, 256, 3, 8), rows(2, 2), False, True,
         [fwd(D3, 2, LSTM, XG), bwd(D3 + M01_SPLIT_KEPT, 2, LSTM, XG, 2, 1, 1)]),
    Case("d3_r3_m01_split", ("lstm", 40, 256, 3, 8), rows(3, 3), True, True,
         [fwd(D3, 3, LSTM, XG), bwd(D3 + M01_SPLIT_KEPT, 3, LSTM, XG, 2, 1, 1)]),
    Case("d3_r4_m01_split", ("lstm", 40, 256, 3, 8), rows(4, 4), False, True,
         [fwd(D3, 4, LSTM, XG), bwd(D3 + M01_SPLIT_KEPT, 4, LSTM, XG, 2, 1, 1)]),
    Case("d3_r5_split", ("lstm", 40, 256, 3, 8), {**rows(5, 1), **THREE_CORE}, True, True,
         [fwd(D3, 5, LSTM, XG), bwd(D3 + SPLIT_KEPT, 1, LSTM, XG, 2, 1)]),
    Case("d3_m01_r1_recompute", ("lstm", 40, 256, 3, 8), {**rows(1, 2), **MERGED_FWD, **RECOMPUTE}, False, True,
         [fwd(D3 + M01, 1, LSTM, XG, 1), bwd(D3, 2, LSTM, XG, 0, 0)]),
    Case("d3_m01_r2_recompute", ("lstm", 40, 256, 3, 8), {**rows(2, 3), **MERGED_FWD, **RECOMPUTE}, True, True,
         [fwd(D3 + M01, 2, LSTM, XG, 1), bwd(D3, 3, LSTM, XG, 0, 0)]),
    Case("d3_m01_r3_kept", ("lstm", 40, 256, 3, 8), {**rows(3, 2), **MERGED_FWD, **FUSED_KEPT}, False, True,
         [fwd(D3 + M01, 3, LSTM, XG, 1), bwd(D3 + KEPT, 2, LSTM, XG, 2, 0)]),
    Case("d3_m01_r4_kept", ("lstm", 40, 256, 3, 8), {**rows(4, 3), **MERGED_FWD, **FUSED_KEPT}, True, True,
         [fwd(D3 + M01, 4, LSTM, XG, 1), bwd(D3 + KEPT, 3, LSTM, XG, 2, 0)]),
    # 256 input features: layer 0 has the ih shape of cfg3's inner layers (TT-matvec kernels with and without dX)
    Case("d3_m01_r5_tt_ih_dx", ("lstm", 256, 256, 3, 8), {**rows(5, 0), **MERGED_FWD, **TT_IH}, True, True,
         [fwd(D3 + M01, 5, LSTM, XG, 1), ttl_fwd("IH_256_H256_d3r8", 4), ttl_bwd("IH_256_H256_d3r8", 3, True)]),
    Case("d3_r2_split_tt_ih", ("lstm", 256, 256, 3, 8), {**rows(0, 2), **THREE_CORE, **TT_IH}, False, True,
         [bwd(D3 + SPLIT_KEPT, 2, LSTM, XG, 2, 1), ttl_bwd("IH_256_H256_d3r8", 3, False)]),
    Case("d3_r3_split_tt_ih", ("lstm", 40, 256, 3, 8), {**rows(0, 3), **THREE_CORE, **TT_IH}, False, True,
         [bwd(D3 + SPLIT_KEPT, 3, LSTM, XG, 2, 1), ttl_fwd("IH_40_H256_d3r8", 8), ttl_bwd("IH_40_H256_d3r8", 4, False)]),
    # H = 768 d2 (the reference's GE2E default width; rank 2 runs rank-padded to 4)
    Case("h768_r2", ("lstm", 40, 768, 2, 2), rows(2, 2), False, True,
         [fwd(H768, 2, LSTM, XG), bwd(H768 + SPLIT_KEPT, 2, LSTM, XG, 2, 1)]),
    Case("h768_r4", ("lstm", 40, 768, 2, 4), rows(4, 3), True, True,
         [fwd(H768, 4, LSTM, XG), bwd(H768 + SPLIT_KEPT, 3, LSTM, XG, 2, 1)]),
    # d4 r16 (cfg4) with the TT-chain ih route
    Case("d4r16_tt_ih", ("lstm", 40, 256, 4, 16), TT_IH, False, True,
         [fwd(D4R16, 1, LSTM, XG), bwd(D4R16 + SPLIT_KEPT, 1, LSTM, XG, 2, 1), ttl_fwd("IH_40_H256_d4r16", 2)]),
    Case("d4r16_tt_ih_256", ("lstm", 256, 256, 4, 16), TT_IH, False, True,
         [ttl_fwd("IH_256_H256_d4r16", 1)]),
    # H = 1024 d4 r8 (cfg5): split BPTT, hh core gradients projected onto the cores by the batched TT-matvec backward
    Case("h1024_tt_ih", ("lstm", 256, 1024, 4, 8), TT_IH, False, True,
         [fwd(H1024, 1, LSTM, XG), bwd(H1024 + SPLIT, 1, LSTM, XG, 0, 1), ttl_fwd("IH_256_H1024_d4r8", 1),
          ttl_bwd("IH_256_H1024_d4r8", 1, False), ttl_bwd("HHW_H1024_d4r8", 1, False)]),
]
LEDGER = {key: case.id for case in CASES for key in case.targets}
KIND_CODE = {"ttl_fwd": 0, "rnn_fwd": 1, "rnn_bwd": 2, "ttl_bwd": 3}       # TTRNN_K_* of the launch records
T_STEPS = 5


def key_id(key):
    kind, name, R, cell, mode, saved, split, merged = key
    return "%s-%s-R%d-c%d-m%d-s%d-p%d-g%d" % (kind, re.sub(r"[^A-Za-z0-9_]+", "_", name).strip("_"), R, cell, mode,
                                               saved, split, merged)


def registry_keys(lib):
    """Registry keys in table order (the order of the launch counters), from ttrnn_static_kernel_keys()."""
    buf = ctypes.create_string_buffer(1 << 16)
    assert lib.ttrnn_static_kernel_keys(buf, len(buf)) > 0
    keys = []
    for ln in buf.value.decode().strip().splitlines():
        c = ln.split("|")
        keys.append((c[0], c[1], int(c[2])) + tuple(int(v) for v in c[3:8]))
    return keys


# ---- running a case --------------------------------------------------------------------------------------------
DEFAULTS = {"chunk_steps": 0, "save_u_bytes": 16 << 30, "static_rows_fwd": 0, "static_rows_bwd": 0, "dense_ih": 1,
            "split_kept": 1, "row_plan": 1, "row_groups": 1, "merge_cores": 1}


@contextmanager
def options(**kw):
    """Library options for the duration of a block; the defaults come back afterwards."""
    from tensorized_rnn_b200 import _lib
    lib = _lib.load()
    for k, v in kw.items():
        assert lib.ttrnn_set_option(k.encode(), int(v)) == 0, k
    try:
        yield lib
    finally:
        for k in kw:
            lib.ttrnn_set_option(k.encode(), DEFAULTS[k])


def case_options(case, **extra):
    return {"row_plan": 0, "row_groups": 0, **case.opts, **extra}


def make_models(case):
    """FP64 oracle layers rounded to FP32, and our module (on the GPU) holding the same values."""
    import tensorized_rnn_b200 as tr
    from helpers import oracle
    from test_gpu_static_paths import _sd_from_layers
    cell, I, H, d, r = case.model
    layers = oracle.random_layers(cell, I, H, 1, d, r, bias=True, seed=123, dtype=torch.float64, scale=1.5)
    for p in oracle.flat_params(layers):
        p.data = p.data.float().double()
        p.requires_grad_(True)
    cls = tr.TTLSTM if cell == "lstm" else tr.TTGRU
    with redirect_stdout(io.StringIO()):
        m = cls(I, H, 1, torch.device("cpu"), n_cores=d, tt_rank=r)
    m.load_state_dict(_sd_from_layers(layers))
    return layers, m.to("cuda:0")


def make_inputs(case, B, T, seed):
    cell, I, H = case.model[:3]
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, T, I, generator=g)
    h0, c0 = 0.5 * torch.randn(B, H, generator=g), 0.5 * torch.randn(B, H, generator=g)
    w = {"out": torch.randn(B, T, H, generator=g), "h": torch.randn(B, H, generator=g),
         "c": torch.randn(B, H, generator=g) if cell == "lstm" else None}
    return x, h0, c0, w


def _loss(res, w):
    loss = (res["out"] * w["out"]).sum() + (res["h"] * w["h"]).sum()
    if w["c"] is not None:
        loss = loss + (res["c"] * w["c"]).sum()
    return loss


def masked(w, first):
    """Upstream weights zeroed on the first `first` batch rows."""
    return {k: (None if v is None else torch.cat([torch.zeros_like(v[:first]), v[first:]])) for k, v in w.items()}


def oracle_run(case, layers, x, h0, c0, ws):
    """FP64 reference: values, and for each upstream weighting in `ws` the gradients wrt params, x, h0, c0."""
    from helpers import oracle
    lstm = case.model[0] == "lstm"
    x64 = x.double().requires_grad_(True)
    h64, c64 = h0.double().requires_grad_(True), c0.double().requires_grad_(True)
    if lstm:
        out, (h, c) = oracle.lstm_forward(layers, x64, (h64, c64))
    else:
        (out, h), c = oracle.gru_forward(layers, x64, h64), None
    res = {"out": out, "h": h, "c": c}
    params = oracle.flat_params(layers)
    wrt = params + [x64, h64] + ([c64] if lstm else [])
    grads = []
    for i, w in enumerate(ws):
        gs = torch.autograd.grad(_loss(res, w), wrt, retain_graph=i + 1 < len(ws))
        n = len(params)
        grads.append({"params": list(gs[:n]), "dx": gs[n], "dh0": gs[n + 1], "dc0": gs[n + 2] if lstm else None})
    return {k: (None if v is None else v.detach()) for k, v in res.items()}, grads


def launch_records(lib):
    n = lib.ttrnn_kernel_launch_records(None, 0)
    buf = (ctypes.c_double * (6 * max(n, 1)))()
    lib.ttrnn_kernel_launch_records(buf, n)
    return [tuple(int(buf[6 * i + j]) for j in range(5)) for i in range(n)]       # kind, R, ctas, rows, steps


def gpu_run(case, m, x, h0, c0, w, lib, train=True, records=False):
    """One step of our module; returns values, gradients, launch counters per registry entry and launch records."""
    lstm = case.model[0] == "lstm"
    dev = "cuda:0"
    ncnt = lib.ttrnn_static_kernel_launches(None, 0, 1)
    kms, kcnt = (ctypes.c_double * 7)(), (ctypes.c_int64 * 7)()
    if records:
        lib.ttrnn_kernel_times(kms, kcnt)
        lib.ttrnn_kernel_timing(1)
    try:
        for p in m.parameters():
            p.grad = None
        xd = x.to(dev).requires_grad_(train and case.xgrad)
        hd, cd = h0.to(dev).requires_grad_(train), c0.to(dev).requires_grad_(train)
        with torch.set_grad_enabled(train):
            out, st = m(xd, (hd, cd) if lstm else hd)
            res = {"out": out, "h": st[0] if lstm else st, "c": st[1] if lstm else None}
            if train:
                _loss(res, {k: (None if v is None else v.to(dev)) for k, v in w.items()}).backward()
        torch.cuda.synchronize()
    finally:
        if records:
            lib.ttrnn_kernel_timing(0)
    recs = []
    if records:
        lib.ttrnn_kernel_times(kms, kcnt)
        recs = launch_records(lib)
    counts = (ctypes.c_int64 * ncnt)()
    lib.ttrnn_static_kernel_launches(counts, ncnt, 1)
    got = {k: (None if v is None else v.detach().cpu()) for k, v in res.items()}
    if train:
        got.update(dx=xd.grad.cpu() if case.xgrad else None, dh0=hd.grad.cpu(), dc0=cd.grad.cpu() if lstm else None,
                   params=[p.grad.cpu() for p in m.flat_parameters()])
    return got, list(counts), recs


def first_round_rows(recs, kinds, B, Rs=None):
    """Batch rows covered by the first round of tiles (tile index < grid) of the matching launches: rows beyond it were
    computed by CTAs that had already run a tile.  TT-matvec rows are (batch row, step) pairs, rows_per_b per batch row;
    launches over other row sets (the projection of dense weight gradients onto the cores) do not count."""
    first = 0
    for kind, R, ctas, nrows, _ in recs:
        if kind not in kinds or R <= 0 or nrows % B or (Rs is not None and (kind, R) not in Rs):
            continue
        rpb = nrows // B
        first = max(first, -(-ctas * R // rpb))
    return min(first, B)


def compare(name, got, ref, first, tol, errs):
    """rel_err over the first-round rows and over the later rows separately."""
    from helpers import rel_err
    if ref is None:
        return
    parts = [("all rows", slice(0, None))] if first in (0, got.shape[0]) else \
        [("first-round rows", slice(0, first)), ("later rows", slice(first, None))]
    for part, sl in parts:
        e = rel_err(got[sl], ref[sl])
        if not e <= tol:
            errs.append("%s over %s: rel err %.2e > %.0e" % (name, part, e, tol))


def compare_step(tag, got, ref, grads, first_f, first_b, errs):
    from helpers import FWD_TOL, GRAD_TOL, rel_err
    for k in ("out", "h", "c"):
        compare("%s %s" % (tag, k), got[k], ref[k], first_f, FWD_TOL, errs)
    for k in ("dx", "dh0", "dc0"):
        if got.get(k) is not None:
            compare("%s %s" % (tag, k), got[k], grads[k], first_b, GRAD_TOL, errs)
    for i, (a, b) in enumerate(zip(got["params"], grads["params"])):
        e = rel_err(a, b)
        if not e <= GRAD_TOL:
            errs.append("%s param %d %s: rel err %.2e" % (tag, i, tuple(b.shape), e))


def batch_sizes(case, sms):
    """Fewer rows than one tile, a ragged last tile within one wave, more tiles than three waves of one CTA per SM (the
    CTAs of a launch loop over tiles; ragged last round).  TT-matvec rows are B x T."""
    rnn_R = [k[2] for k in case.targets if k[0].startswith("rnn")] or [1]
    ttl_R = [k[2] for k in case.targets if k[0].startswith("ttl")]
    R = max(rnn_R + [max(case.opts.get("static_rows_fwd", 1), case.opts.get("static_rows_bwd", 1))])
    big = 3 * sms * R + (R + 1) // 2
    for Rt in ttl_R:
        big = max(big, -(-(3 * sms * Rt + (Rt + 1) // 2) // T_STEPS) | 1)
    small = [B for B in (R - 1, 3 * R + 1) if B >= 1]
    return small, big


_REPORTS = {}


def case_report(case_id):
    """Runs a case once (shared by the tests of its registry keys): errors, per-key launch evidence, describe."""
    if case_id in _REPORTS:
        return _REPORTS[case_id]
    from tensorized_rnn_b200 import _lib
    case = next(c for c in CASES if c.id == case_id)
    lib = _lib.load()
    keys = registry_keys(lib)
    idx = {k: i for i, k in enumerate(keys)}
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    T = T_STEPS
    rep = {"errors": [], "missed": [], "rounds": {}, "describe": {}}
    layers, m = make_models(case)
    small, big = batch_sizes(case, sms)
    tkeys = [k for k in case.targets if k in idx]
    rep["missed"] += ["not in the registry: %r" % (k,) for k in case.targets if k not in idx]

    def counted(tag, counts, B, Tc):
        for k in tkeys:
            if k[0].startswith("ttl") and B * Tc < 64:
                continue                                 # tiny TT-matvec calls stay on the runtime-shape kernel
            if counts[idx[k]] < 1:
                rep["missed"].append("%s: %s did not launch" % (tag, key_id(k)))

    with options(**case_options(case)) as lib:
        for B in small + [big]:
            x, h0, c0, w = make_inputs(case, B, T, seed=B)
            is_big = B == big
            got, counts, recs = gpu_run(case, m, x, h0, c0, w, lib, records=True)
            counted("B=%d" % B, counts, B, T)
            first_f = first_round_rows(recs, (0, 1), B, {(KIND_CODE[k[0]], k[2]) for k in tkeys if k[0] == "ttl_fwd"}
                                       | {(1, r[1]) for r in recs if r[0] == 1})
            first_b = first_round_rows(recs, (2, 3), B, {(KIND_CODE[k[0]], k[2]) for k in tkeys if k[0] == "ttl_bwd"}
                                       | {(2, r[1]) for r in recs if r[0] == 2})
            first = max(first_f, first_b)
            if is_big:
                for k in tkeys:
                    tiles = [(-(-r[3] // r[1]), r[2]) for r in recs if r[0] == KIND_CODE[k[0]] and r[1] == k[2]]
                    rep["rounds"][k] = max([t / c for t, c in tiles if c > 0], default=0.0)
                if not first < B:
                    rep["errors"].append("B=%d: no rows beyond the first round of tiles (records %r)" % (B, recs))
            ws = [w, masked(w, first)] if is_big else [w]
            ref, grads = oracle_run(case, layers, x, h0, c0, ws)
            compare_step("B=%d" % B, got, ref, grads[0], first_f, first_b, rep["errors"])
            if is_big:
                # parameter gradients made only by rows that CTAs ran after their first tile
                got2, _, _ = gpu_run(case, m, x, h0, c0, masked(w, first), lib)
                from helpers import GRAD_TOL, rel_err
                for i, (a, b) in enumerate(zip(got2["params"], grads[1]["params"])):
                    e = rel_err(a, b)
                    if not e <= GRAD_TOL:
                        rep["errors"].append("B=%d later-round rows only: param %d %s rel err %.2e"
                                             % (B, i, tuple(b.shape), e))
                # inference takes the saved == NULL branch of the forward kernels: bit-identical results
                inf, counts, _ = gpu_run(case, m, x, h0, c0, w, lib, train=False)
                for k in ("out", "h", "c"):
                    if got[k] is not None and not torch.equal(inf[k], got[k]):
                        rep["errors"].append("B=%d: no_grad forward %s differs from the training forward" % (B, k))
                for k in tkeys:
                    if k[0].endswith("fwd") and counts[idx[k]] < 1:
                        rep["missed"].append("no_grad: %s did not launch" % key_id(k))
                plan = _lib.describe_plan(m.spec().desc(B, T), training=True)[1]
                rep["describe"] = plan
                if case.chunk:
                    # time chunks of 2 steps (2, 2, 1): per-chunk row offsets, states handed between launches
                    with options(chunk_steps=2):
                        got3, counts, recs3 = gpu_run(case, m, x, h0, c0, w, lib, records=True)
                    counted("chunk_steps=2", counts, B, 2)
                    f3 = first_round_rows(recs3, (1,), B)
                    b3 = first_round_rows(recs3, (2,), B)
                    compare_step("chunk_steps=2", got3, ref, grads[0], f3, b3, rep["errors"])
    _REPORTS[case_id] = rep
    return rep


def _check_key(key):
    rep = case_report(LEDGER[key])
    assert not rep["missed"], rep["missed"]
    assert not rep["errors"], rep["errors"]
    kind, name, R = key[:3]
    # the CTAs of the large batch looped over more than one tile
    print("%s: tiles / CTAs = %.2f" % (key_id(key), rep["rounds"].get(key, 0.0)))
    assert rep["rounds"].get(key, 0.0) > 1.0, "tiles / CTAs = %r" % rep["rounds"].get(key)
    plan, tok = rep["describe"], name.replace(" ", "_")
    if kind == "rnn_fwd":
        assert (plan["fwd_kernel"], plan["fwd_rows"]) == (tok, R), plan
    elif kind == "rnn_bwd":
        assert (plan["bwd_kernel"], plan["bwd_rows"]) == (tok, R), plan


KEYS = sorted(LEDGER)


@pytest.mark.parametrize("key", KEYS, ids=[key_id(k) for k in KEYS])
def test_static_kernel_matches_fp64_oracle(key):
    _check_key(key)


# ---- rank-one input with dX (the projected-input BPTT route of layer 0) -----------------------------------------------
RANK1_DX = [
    # id, (cell, I, H, d, r): a chunked plan (chunk_steps = 4, T = 9) rules out the rank-one split kernels
    ("lstm_d2r4", ("lstm", 1, 256, 2, 4)),
    ("lstm_d2r3_rank_padded", ("lstm", 1, 256, 2, 3)),
    ("gru_d2r4", ("gru", 1, 256, 2, 4)),
]


@pytest.mark.parametrize("case", RANK1_DX, ids=[c[0] for c in RANK1_DX])
def test_rank_one_input_gradient_route_matches_oracle(case):
    """A rank-one layer 0 whose input gradient is requested runs the projected-input BPTT kernels.  The workspace must be
    sized for them also when the rank-one split route does not apply (chunked plans): the LSTM then takes the
    dX-only kernel with its dense hh-gradient buffers, the GRU the fused kept-gates kernel.  describe names that kernel
    as bwd_kernel_dx."""
    from tensorized_rnn_b200 import _lib
    name, model = case
    c = Case(name, model, {"chunk_steps": 4}, True, False, [])
    T = 9
    lib = _lib.load()
    keys = registry_keys(lib)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = 3 * sms * 4 + 2
    layers, m = make_models(c)
    x, h0, c0, w = make_inputs(c, B, T, seed=3)
    with options(**case_options(c)) as lib:
        plan = _lib.describe_plan(m.spec().desc(B, T), training=True)[1]
        got, counts, recs = gpu_run(c, m, x, h0, c0, w, lib, records=True)
    assert plan["ih_route"] == "rank_one" and "bwd_kernel_dx" in plan, plan
    ran = [k for k, n in zip(keys, counts) if n > 0 and k[0] == "rnn_bwd"]
    assert len(ran) == 1 and ran[0][4] == XG, ran
    assert (ran[0][1].replace(" ", "_"), ran[0][2]) == (plan["bwd_kernel_dx"], plan["bwd_rows_dx"]), (ran, plan)
    if model[0] == "lstm":
        assert ran[0][5:7] == (2, 1), ran                 # kept gates, dX-only kernel + dense hh core gradients
    else:
        assert ran[0][5:7] == (2, 0), ran                 # no split GRU variant behind a projected input
    assert any(r[0] == 2 and -(-r[3] // r[1]) > r[2] for r in recs), recs
    first_f = first_round_rows(recs, (1,), B)
    first_b = first_round_rows(recs, (2,), B)
    ref, grads = oracle_run(c, layers, x, h0, c0, [w])
    errs = []
    compare_step("B=%d" % B, got, ref, grads[0], first_f, first_b, errs)
    assert not errs, errs
