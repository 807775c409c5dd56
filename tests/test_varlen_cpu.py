"""Variable-length rows (DESIGN.md §4.22) without a GPU: the references against each other, the frozen-gate argument in
float32, validation, and the C ABI (new symbols, the plan flag refused by every other entry point)."""
import ctypes as C
import os

import numpy as np
import pytest
import torch
from torch.nn.utils.rnn import pack_padded_sequence, pad_packed_sequence

import tensorized_rnn_b200 as tr
from tensorized_rnn_b200 import _lib
from tensorized_rnn_b200.functional import check_lengths, pack_like, unpack_sequence
from helpers import ROOT, oracle
from varlen_ref import oracle_rows, torch_packed

CPU = torch.device("cpu")


@pytest.mark.parametrize("cell", ["lstm", "gru"])
@pytest.mark.parametrize("L,init", [(1, False), (2, True), (3, False)])
def test_oracle_rows_match_torch_packed(cell, L, init):
    layers = oracle.random_layers(cell, 12, 16, L, 2, 3, seed=3 + L, dtype=torch.float64)
    g = torch.Generator().manual_seed(4)
    lengths = [5, 1, 7, 3, 7, 2]
    x = torch.randn(len(lengths), 7, 12, generator=g, dtype=torch.float64)
    B, H = len(lengths), 16
    st = None
    if init:
        st = tuple(torch.randn(B, H, generator=g, dtype=torch.float64) for _ in range(2 if cell == "lstm" else 1))
        st = st if cell == "lstm" else st[0]
    a = oracle_rows(cell, layers, x, lengths, st)
    b = torch_packed(cell, layers, x, lengths, st)
    for u, v in zip(a, b):
        assert (u - v).abs().max().item() <= 1e-12


def _sig(v):
    return np.float32(1) / (np.float32(1) + np.exp(-v, dtype=np.float32))


def test_gates_freeze_bit_exactly_at_infinity():
    """The frozen ih columns (LSTM i = -inf, f = +inf, g = o = 0; GRU z = +inf, r = n = 0) give exact 0 / 1 gates in
    float32 for any finite hh part, so c_t (LSTM) and h_t (GRU) are carried bit for bit and every gate delta is 0."""
    rng = np.random.default_rng(0)
    with np.errstate(over="ignore"):
        u = (rng.standard_normal(4096) * 30).astype(np.float32)
        c_prev = (rng.standard_normal(4096) * 5).astype(np.float32)
        h_prev = rng.standard_normal(4096).astype(np.float32)
        i, f = _sig(np.float32(-np.inf) + u), _sig(np.float32(np.inf) + u)
        g, o = np.tanh(np.float32(0) + u), _sig(np.float32(0) + u)
        assert (i == 0).all() and (f == 1).all()
        c = f * c_prev + i * g
        assert np.array_equal(c, c_prev)
        dc = rng.standard_normal(4096).astype(np.float32)
        assert (dc * g * i * (1 - i) == 0).all() and (dc * c_prev * f * (1 - f) == 0).all() and (dc * i * (1 - g * g) == 0).all()
        assert np.array_equal(dc * f, dc)
        z = _sig(np.float32(np.inf) + u)
        r = _sig(np.float32(0) + u)
        n = np.tanh(np.float32(0) + r * u)
        assert (z == 1).all()
        assert np.array_equal((1 - z) * n + z * h_prev, h_prev)
        dh = rng.standard_normal(4096).astype(np.float32)
        assert (dh * (1 - z) == 0).all() and (dh * (h_prev - n) * z * (1 - z) == 0).all()


def test_lengths_validation():
    assert check_lengths([3, 1, 4], 3, 4, CPU).tolist() == [3, 1, 4]
    assert check_lengths(torch.tensor([4, 4]), 2, 4, CPU).dtype == torch.int32
    for bad, why in (([0, 2], "0"), ([2, 5], "above T"), ([1, 2, 3], "count"), ([1.0, 2.0], "float"), ([[1, 2]], "2-D")):
        with pytest.raises(ValueError):
            check_lengths(bad, 2, 4, CPU)


def test_unsorted_packed_sequence_round_trip():
    g = torch.Generator().manual_seed(1)
    lengths = torch.tensor([2, 5, 5, 1, 3])
    x = torch.randn(5, 5, 3, generator=g)
    packed = pack_padded_sequence(x, lengths, batch_first=True, enforce_sorted=False)
    padded, lens = unpack_sequence(packed)
    assert lens.tolist() == lengths.tolist()
    assert torch.equal(padded, x * (torch.arange(5)[None, :, None] < lengths[:, None, None]))
    back = pack_like(padded * 2, lens, packed)
    assert torch.equal(back.batch_sizes, packed.batch_sizes)
    assert torch.equal(back.sorted_indices, packed.sorted_indices)
    assert torch.equal(back.unsorted_indices, packed.unsorted_indices)
    assert torch.equal(back.data, packed.data * 2)
    srt = pack_padded_sequence(x[[1, 2, 4, 0, 3]], lengths[[1, 2, 4, 0, 3]], batch_first=True)
    assert pack_like(unpack_sequence(srt)[0], unpack_sequence(srt)[1], srt).sorted_indices is None


@pytest.mark.parametrize("kw", [dict(is_naive=True), dict(log_grads=True)])
def test_cell_step_mode_refuses_packed_input(kw):
    m = tr.TTLSTM(8, 16, 1, CPU, n_cores=2, tt_rank=2, **kw)
    packed = pack_padded_sequence(torch.zeros(2, 3, 8), torch.tensor([3, 2]), batch_first=True)
    with pytest.raises(NotImplementedError):
        m(packed)
    with pytest.raises(NotImplementedError):
        m.forward_states(packed)


NEW = ["ttrnn_rnn_forward_lengths", "ttrnn_rnn_backward_lengths", "ttrnn_dense_rnn_forward_lengths",
       "ttrnn_dense_rnn_backward_lengths", "ttrnn_time_reverse_add_lengths", "ttrnn_bidir_join_lengths",
       "ttrnn_rnn_describe_ex"]


def test_new_symbols_are_declared_and_exported():
    header = open(os.path.join(ROOT, "include", "ttrnn_b200.h")).read()
    lib = _lib.load()
    assert "#define TTRNN_WS_LENGTHS 16" in header and _lib.WS_LENGTHS == 16
    for name in NEW:
        assert name + "(" in header and name in _lib.SYMBOLS
        assert getattr(lib, name) is not None
    assert lib.ttrnn_abi_version() == 4


def _plan(entry_bits):
    """A workspace struct as ttrnn_rnn_workspace_bytes_ex stamps it, with the entry-point word set (the sizing call itself
    needs a device): magic, then the option snapshot, group count, rows, layer states, dropout, entry bits."""
    ws = _lib.RnnWorkspace()
    ws.plan[0] = 0x7474726E6E706C36
    ws.plan[_lib.PLAN_WORDS - 1] = entry_bits
    return ws


def _desc():
    d = _lib.RnnDesc()
    d.cell, d.num_layers, d.input_size, d.hidden_size, d.has_bias, d.seq_len, d.batch = 0, 1, 4, 4, 1, 3, 2
    return d


def test_old_entry_points_refuse_a_lengths_plan():
    lib = _lib.load()
    d, ws = _desc(), _plan(2)
    calls = {
        "ttrnn_rnn_forward": lambda: lib.ttrnn_rnn_forward(C.byref(d), C.byref(ws), *([None] * 9), None),
        "ttrnn_rnn_forward_dropout": lambda: lib.ttrnn_rnn_forward_dropout(C.byref(d), C.byref(ws), *([None] * 10), None),
        "ttrnn_rnn_forward_proj": lambda: lib.ttrnn_rnn_forward_proj(C.byref(d), C.byref(ws), *([None] * 10), None, None),
        "ttrnn_rnn_backward": lambda: lib.ttrnn_rnn_backward(C.byref(d), C.byref(ws), *([None] * 15)),
        "ttrnn_rnn_backward_dropout": lambda: lib.ttrnn_rnn_backward_dropout(C.byref(d), C.byref(ws), *([None] * 16)),
        "ttrnn_rnn_backward_proj": lambda: lib.ttrnn_rnn_backward_proj(C.byref(d), C.byref(ws), *([None] * 17)),
        "ttrnn_rnn_backward_logged": lambda: lib.ttrnn_rnn_backward_logged(C.byref(d), C.byref(ws), *([None] * 15),
                                                                           C.c_void_p(16), None),
        "ttrnn_rnn_saved_layout": lambda: lib.ttrnn_rnn_saved_layout(C.byref(d), C.byref(ws), 0, C.byref(C.c_int64()),
                                                                     C.byref(C.c_int64())),
    }
    for name, call in calls.items():
        assert call() != 0, name
        assert "TTRNN_WS_LENGTHS" in _lib.last_error(), (name, _lib.last_error())


def test_lengths_entry_points_refuse_a_plan_without_the_flag():
    lib = _lib.load()
    d = _desc()
    one = (C.c_int32 * 2)(3, 3)
    for ws in (_plan(0), _plan(1)):
        pj = C.byref(_lib.RnnProj()) if ws.plan[_lib.PLAN_WORDS - 1] else None
        assert lib.ttrnn_rnn_forward_lengths(C.byref(d), C.byref(ws), *([None] * 10), pj, None, C.addressof(one)) != 0
        assert "TTRNN_WS_LENGTHS" in _lib.last_error()
        assert lib.ttrnn_rnn_backward_lengths(C.byref(d), C.byref(ws), *([None] * 15), pj, None, C.addressof(one)) != 0
        assert "TTRNN_WS_LENGTHS" in _lib.last_error()
    ws = _plan(2)
    assert lib.ttrnn_rnn_forward_lengths(C.byref(d), C.byref(ws), *([None] * 10), None, None, None) != 0
    assert "lengths must be non-null" in _lib.last_error()
    assert lib.ttrnn_rnn_forward_lengths(C.byref(d), C.byref(ws), *([None] * 10), C.byref(_lib.RnnProj()), None,
                                         C.addressof(one)) != 0
    assert "pj must be given exactly" in _lib.last_error()
    dd = _lib.DenseDesc(0, 1, 128, 128, 1, 3, 2)
    assert lib.ttrnn_dense_rnn_forward_lengths(C.byref(dd), *([None] * 10), 0, 0, None) != 0
    assert "lengths must be non-null" in _lib.last_error()
    assert lib.ttrnn_dense_rnn_forward_ex(C.byref(dd), *([None] * 10), _lib.WS_LENGTHS) != 0
    assert "unknown flags" in _lib.last_error()
