"""ctypes binding of the C ABI in include/ttrnn_b200.h.

The shared library is built in-tree by `tensorized_rnn_b200.build`.  There is no
fallback of any kind: if the library is missing, or a compute entry point is called
without a CUDA device / with CPU tensors, the call raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

ABI_VERSION = 4
MAX_CORES = 6
MAX_LAYERS = 8
PLAN_WORDS = 24
WS_WHOLE_BATCH = 1
WS_LAYER_STATES = 2      # per-layer (L, B, H) initial / final states and their gradients
WS_DROPOUT = 4           # inter-layer dropout: saved keeps the masked inputs of layers 1 .. L-1
WS_PROJ = 8              # projected LSTM (proj_size): the plan of the _proj entry points
WS_LENGTHS = 16          # variable-length rows: the plan of the _lengths entry points
CELL_LSTM, CELL_GRU = 0, 1

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "libttrnn_b200.so")
_lib: Optional[C.CDLL] = None


class TTShape(C.Structure):
    _fields_ = [("d", C.c_int32),
                ("in_modes", C.c_int32 * MAX_CORES),
                ("out_modes", C.c_int32 * MAX_CORES),
                ("ranks", C.c_int32 * (MAX_CORES + 1))]


class RnnDesc(C.Structure):
    _fields_ = [("cell", C.c_int32), ("num_layers", C.c_int32), ("input_size", C.c_int32),
                ("hidden_size", C.c_int32), ("has_bias", C.c_int32), ("seq_len", C.c_int32),
                ("batch", C.c_int64),
                ("ih", TTShape * MAX_LAYERS), ("hh", TTShape * MAX_LAYERS)]


class DenseDesc(C.Structure):
    _fields_ = [("cell", C.c_int32), ("num_layers", C.c_int32), ("input_size", C.c_int32), ("hidden_size", C.c_int32),
                ("has_bias", C.c_int32), ("seq_len", C.c_int32), ("batch", C.c_int64)]


class RnnWorkspace(C.Structure):
    # `plan`: opaque execution plan stamped by ttrnn_rnn_workspace_bytes(); the same struct goes to the forward and
    # to its backward so both interpret `saved` / scratch identically whatever happens to the options in between
    _fields_ = [("saved_bytes", C.c_int64), ("fwd_scratch_bytes", C.c_int64), ("bwd_scratch_bytes", C.c_int64),
                ("plan", C.c_int64 * PLAN_WORDS)]


class Dropout(C.Structure):
    _fields_ = [("p", C.c_float), ("reserved", C.c_int32), ("seed", C.c_uint64), ("offset", C.c_uint64)]


class RnnProj(C.Structure):
    _fields_ = [("proj_size", C.c_int32), ("reserved", C.c_int32), ("hr", TTShape * MAX_LAYERS)]


# every symbol include/ttrnn_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "ttrnn_abi_version": (C.c_int, []),
    "ttrnn_last_error": (C.c_char_p, []),
    "ttrnn_rnn_param_count": (C.c_int64, [C.POINTER(RnnDesc)]),
    "ttrnn_rnn_workspace_bytes": (C.c_int, [C.POINTER(RnnDesc), C.POINTER(RnnWorkspace)]),
    "ttrnn_rnn_workspace_bytes_ex": (C.c_int, [C.POINTER(RnnDesc), C.c_int32, C.POINTER(RnnWorkspace)]),
    "ttrnn_rnn_saved_layout": (C.c_int, [C.POINTER(RnnDesc), C.POINTER(RnnWorkspace), C.c_int32, C.POINTER(C.c_int64),
                                         C.POINTER(C.c_int64)]),
    "ttrnn_rnn_backward_logged": (C.c_int, [C.POINTER(RnnDesc), C.POINTER(RnnWorkspace)] + [_P] * 17),
    "ttrnn_step_norms": (C.c_int, [_P, C.c_int64, C.c_int32, C.c_int32, _P, _P]),
    "ttrnn_time_reverse_add": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "ttrnn_bidir_join": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    "ttrnn_rnn_forward": (C.c_int, [C.POINTER(RnnDesc), C.POINTER(RnnWorkspace)] + [_P] * 10),
    "ttrnn_rnn_backward": (C.c_int, [C.POINTER(RnnDesc), C.POINTER(RnnWorkspace)] + [_P] * 15),
    "ttrnn_rnn_forward_dropout": (C.c_int, [C.POINTER(RnnDesc), C.POINTER(RnnWorkspace)] + [_P] * 10 + [C.POINTER(Dropout)]),
    "ttrnn_rnn_backward_dropout": (C.c_int, [C.POINTER(RnnDesc), C.POINTER(RnnWorkspace)] + [_P] * 15 +
                                   [C.POINTER(Dropout)]),
    "ttrnn_rnn_param_count_proj": (C.c_int64, [C.POINTER(RnnDesc), C.POINTER(RnnProj)]),
    "ttrnn_rnn_workspace_bytes_proj": (C.c_int, [C.POINTER(RnnDesc), C.POINTER(RnnProj), C.c_int32, C.POINTER(RnnWorkspace)]),
    "ttrnn_rnn_forward_proj": (C.c_int, [C.POINTER(RnnDesc), C.POINTER(RnnWorkspace)] + [_P] * 10 +
                               [C.POINTER(RnnProj), C.POINTER(Dropout)]),
    "ttrnn_rnn_backward_proj": (C.c_int, [C.POINTER(RnnDesc), C.POINTER(RnnWorkspace)] + [_P] * 15 +
                                [C.POINTER(RnnProj), C.POINTER(Dropout)]),
    "ttrnn_rnn_forward_lengths": (C.c_int, [C.POINTER(RnnDesc), C.POINTER(RnnWorkspace)] + [_P] * 10 +
                                  [C.POINTER(RnnProj), C.POINTER(Dropout), _P]),
    "ttrnn_rnn_backward_lengths": (C.c_int, [C.POINTER(RnnDesc), C.POINTER(RnnWorkspace)] + [_P] * 15 +
                                   [C.POINTER(RnnProj), C.POINTER(Dropout), _P]),
    "ttrnn_time_reverse_add_lengths": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    "ttrnn_bidir_join_lengths": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "ttrnn_dropout_apply": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.POINTER(Dropout),
                                      _P, _P, _P, _P]),
    "ttrnn_ttlinear_param_count": (C.c_int64, [C.POINTER(TTShape)]),
    "ttrnn_ttlinear_workspace_bytes": (C.c_int64, [C.POINTER(TTShape), C.c_int64]),
    "ttrnn_ttlinear_forward": (C.c_int, [C.POINTER(TTShape), C.c_int64] + [_P] * 6),
    "ttrnn_ttlinear_backward": (C.c_int, [C.POINTER(TTShape), C.c_int64] + [_P] * 8),
    "ttrnn_cell_forward": (C.c_int, [C.c_int32, C.c_int64, C.c_int32] + [_P] * 7),
    "ttrnn_cell_backward": (C.c_int, [C.c_int32, C.c_int64, C.c_int32] + [_P] * 12),
    "ttrnn_dense_rnn_param_count": (C.c_int64, [C.POINTER(DenseDesc)]),
    "ttrnn_dense_rnn_workspace_bytes": (C.c_int, [C.POINTER(DenseDesc), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "ttrnn_dense_rnn_forward": (C.c_int, [C.POINTER(DenseDesc)] + [_P] * 10),
    "ttrnn_dense_rnn_backward": (C.c_int, [C.POINTER(DenseDesc)] + [_P] * 15),
    "ttrnn_dense_rnn_forward_ex": (C.c_int, [C.POINTER(DenseDesc)] + [_P] * 10 + [C.c_int32]),
    "ttrnn_dense_rnn_backward_ex": (C.c_int, [C.POINTER(DenseDesc)] + [_P] * 15 + [C.c_int32]),
    "ttrnn_dense_rnn_param_count_proj": (C.c_int64, [C.POINTER(DenseDesc), C.c_int32]),
    "ttrnn_dense_rnn_workspace_bytes_proj": (C.c_int, [C.POINTER(DenseDesc), C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                                       C.c_int32]),
    "ttrnn_dense_rnn_forward_proj": (C.c_int, [C.POINTER(DenseDesc)] + [_P] * 10 + [C.c_int32, C.c_int32]),
    "ttrnn_dense_rnn_backward_proj": (C.c_int, [C.POINTER(DenseDesc)] + [_P] * 15 + [C.c_int32, C.c_int32]),
    "ttrnn_dense_rnn_forward_lengths": (C.c_int, [C.POINTER(DenseDesc)] + [_P] * 10 + [C.c_int32, C.c_int32, _P]),
    "ttrnn_dense_rnn_backward_lengths": (C.c_int, [C.POINTER(DenseDesc)] + [_P] * 15 + [C.c_int32, C.c_int32, _P]),
    "ttrnn_embed_forward": (C.c_int, [C.c_int64, C.c_int32] + [_P] * 4),
    "ttrnn_embed_backward": (C.c_int, [C.c_int64, C.c_int32] + [_P] * 6),
    "ttrnn_ge2e_workspace_bytes": (C.c_int64, [C.c_int32, C.c_int32, C.c_int32]),
    "ttrnn_ge2e_loss_forward": (C.c_int, [C.c_int32, C.c_int32, C.c_int32] + [_P] * 6),
    "ttrnn_ge2e_loss_backward": (C.c_int, [C.c_int32, C.c_int32, C.c_int32] + [_P] * 7),
    "ttrnn_partials_gather": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, _P, C.c_int64, _P, _P, _P, _P]),
    "ttrnn_segment_mean_normalize_forward": (C.c_int, [C.c_int64, C.c_int32] + [_P] * 5),
    "ttrnn_segment_mean_normalize_backward": (C.c_int, [C.c_int64, C.c_int32] + [_P] * 6),
    "ttrnn_rnn_ih_route": (C.c_int, [C.POINTER(RnnDesc), C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "ttrnn_static_kernel_table": (C.c_int, [C.c_char_p, C.c_int32]),
    "ttrnn_static_kernel_keys": (C.c_int, [C.c_char_p, C.c_int32]),
    "ttrnn_rnn_describe": (C.c_int, [C.POINTER(RnnDesc), C.c_int32, C.c_char_p, C.c_int32]),
    "ttrnn_rnn_describe_ex": (C.c_int, [C.POINTER(RnnDesc), C.c_int32, C.c_int32, C.c_char_p, C.c_int32]),
    "ttrnn_tc_launch_count": (C.c_int64, [C.c_int32]),
    "ttrnn_static_kernel_launches": (C.c_int, [C.POINTER(C.c_int64), C.c_int32, C.c_int32]),
    "ttrnn_rnn_row_groups": (C.c_int, [C.POINTER(RnnDesc), C.c_int32, C.POINTER(C.c_int64)]),
    "ttrnn_ffma_probe": (C.c_int, [C.c_int32, _P, C.POINTER(C.c_double), _P]),
    "ttrnn_launch_count": (C.c_int64, [C.c_int32]),
    "ttrnn_kernel_timing": (C.c_int, [C.c_int32]),
    "ttrnn_kernel_times": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "ttrnn_kernel_launch_records": (C.c_int64, [C.POINTER(C.c_double), C.c_int64]),
    "ttrnn_set_option": (C.c_int, [C.c_char_p, C.c_int64]),
}


def lib_path() -> str:
    return _LIB_PATH


def load() -> C.CDLL:
    """Load the CUDA library; raise loudly if it is not there."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise RuntimeError(
            "tensorized_rnn_b200: CUDA library %s is missing. Build it with "
            "`python -m tensorized_rnn_b200.build` (needs nvcc). There is no CPU or PyTorch fallback." % _LIB_PATH)
    lib = C.CDLL(_LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    if lib.ttrnn_abi_version() != ABI_VERSION:
        raise RuntimeError("tensorized_rnn_b200: ABI version mismatch between %s and the Python binding" % _LIB_PATH)
    for key, env in (("rows_per_cta", "TTRNN_ROWS_PER_CTA"), ("chunk_steps", "TTRNN_CHUNK_STEPS"),
                     ("chunk_bytes", "TTRNN_CHUNK_BYTES"), ("static_rows_fwd", "TTRNN_STATIC_ROWS_FWD"),
                     ("static_rows_bwd", "TTRNN_STATIC_ROWS_BWD"), ("static_kernels", "TTRNN_STATIC_KERNELS"),
                     ("dense_ih", "TTRNN_DENSE_IH"), ("dense_ih_ratio", "TTRNN_DENSE_IH_RATIO"),
                     ("save_u_bytes", "TTRNN_SAVE_U_BYTES"),
                     ("row_plan", "TTRNN_ROW_PLAN"), ("gemm_wide", "TTRNN_GEMM_WIDE"), ("split_kept", "TTRNN_SPLIT_KEPT"),
                     ("dense_hh_dw", "TTRNN_DENSE_HH_DW"), ("tc_gemm", "TTRNN_TC_GEMM"),
                     ("rank_pad", "TTRNN_RANK_PAD"), ("bwd_overlap", "TTRNN_BWD_OVERLAP"),
                     ("row_groups", "TTRNN_ROW_GROUPS"), ("merge_cores", "TTRNN_MERGE_CORES")):
        if os.environ.get(env):
            lib.ttrnn_set_option(key.encode(), int(os.environ[env]))
    _lib = lib
    return lib


def describe_plan(desc: "RnnDesc", training: bool = True, flags: int = 0) -> list:
    """Execution plan of a descriptor (ttrnn_rnn_describe) as a list of dicts: [header, layer 0, layer 1, ...].
    flags: the workspace flags of the plan (ttrnn_rnn_describe_ex), e.g. WS_LENGTHS."""
    lib = load()
    buf = C.create_string_buffer(8192)
    if flags:
        n = lib.ttrnn_rnn_describe_ex(C.byref(desc), int(flags), 1 if training else 0, buf, 8192)
    else:
        n = lib.ttrnn_rnn_describe(C.byref(desc), 1 if training else 0, buf, 8192)
    if n < 0:
        raise RuntimeError("ttrnn_rnn_describe failed: " + last_error())
    out = []
    for line in buf.value.decode().strip().split("\n"):
        ent = {}
        for tok in line.split():
            k, _, v = tok.partition("=")
            ent[k] = int(v) if v.lstrip("-").isdigit() else v
        out.append(ent)
    return out


def last_error() -> str:
    return load().ttrnn_last_error().decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError("%s failed: %s" % (what, last_error()))


def make_tt_shape(in_modes: Sequence[int], out_modes: Sequence[int], ranks: Sequence[int]) -> TTShape:
    d = len(in_modes)
    if d > MAX_CORES:
        raise ValueError("at most %d TT cores are supported, got %d" % (MAX_CORES, d))
    if len(out_modes) != d or len(ranks) != d + 1:
        raise ValueError("inconsistent TT shape: in %r out %r ranks %r" % (in_modes, out_modes, ranks))
    s = TTShape()
    s.d = d
    for k in range(d):
        s.in_modes[k] = int(in_modes[k])
        s.out_modes[k] = int(out_modes[k])
    for k in range(d + 1):
        s.ranks[k] = int(ranks[k])
    return s
