"""Per-layer states without a GPU: the per-layer reference the GPU tests compare against (tests/layer_states_ref.py, the
oracle run one layer at a time) and the C-ABI surface of the feature (TTRNN_WS_LAYER_STATES,
ttrnn_dense_rnn_forward_ex / _backward_ex)."""
import io
import os
import re
from contextlib import redirect_stdout

import pytest
import torch

from tensorized_rnn_b200 import _lib
from helpers import ROOT, oracle
from layer_states_ref import gru_layer_states, lstm_layer_states

CELLS = [("lstm", 12, 20, 3, 2, 3), ("gru", 10, 16, 2, 2, 2)]


def _layers(cell, I, H, L, d, r):
    return oracle.random_layers(cell, I, H, L, d, r, seed=4, dtype=torch.float64, scale=1.5)


def _per_layer(cell, layers, x, states):
    if cell == "lstm":
        return lstm_layer_states(oracle.lstm_forward, layers, x, states)
    return gru_layer_states(oracle.gru_forward, layers, x, None if states is None else states[0])


@pytest.mark.parametrize("case", CELLS, ids=[c[0] for c in CELLS])
def test_per_layer_reference_with_broadcast_states_equals_the_shared_oracle(case):
    cell, I, H, L, d, r = case
    layers = _layers(*case)
    g = torch.Generator().manual_seed(1)
    B, T = 3, 5
    x = torch.rand(B, T, I, generator=g, dtype=torch.float64)
    s = [torch.randn(B, H, generator=g, dtype=torch.float64) for _ in range(2 if cell == "lstm" else 1)]
    if cell == "lstm":
        out_s, fin_s = oracle.lstm_forward(layers, x, tuple(s))
        fin_s = list(fin_s)
    else:
        out_s, h = oracle.gru_forward(layers, x, s[0])
        fin_s = [h]
    out_l, fin_l = _per_layer(cell, layers, x, [v.expand(L, B, H) for v in s])
    assert torch.allclose(out_s, out_l, rtol=0, atol=1e-14)
    for a, b in zip(fin_s, fin_l):
        assert b.shape == (L, B, H) and torch.allclose(a, b[L - 1], rtol=0, atol=1e-14)
    out_0, fin_0 = _per_layer(cell, layers, x, None)                 # no states: zeros
    assert torch.allclose(out_0, (oracle.lstm_forward if cell == "lstm" else oracle.gru_forward)(layers, x)[0],
                          rtol=0, atol=1e-14)
    assert fin_0[0].shape == (L, B, H)


@pytest.mark.parametrize("case", CELLS, ids=[c[0] for c in CELLS])
def test_final_layer_states_continue_the_sequence(case):
    """The per-layer final states of a run over the first steps, fed into a run over the remaining steps, give the
    outputs and final states of one run over the whole sequence."""
    cell, I, H, L, d, r = case
    layers = _layers(*case)
    g = torch.Generator().manual_seed(2)
    B, T, cut = 3, 7, 3
    x = torch.rand(B, T, I, generator=g, dtype=torch.float64)
    s = [torch.randn(L, B, H, generator=g, dtype=torch.float64) for _ in range(2 if cell == "lstm" else 1)]
    out, fin = _per_layer(cell, layers, x, s)
    out_a, fin_a = _per_layer(cell, layers, x[:, :cut], s)
    out_b, fin_b = _per_layer(cell, layers, x[:, cut:], fin_a)
    assert torch.allclose(torch.cat([out_a, out_b], dim=1), out, rtol=0, atol=1e-14)
    for a, b in zip(fin_b, fin):
        assert torch.allclose(a, b, rtol=0, atol=1e-14)
    # the inner layers' final states matter: carrying only the last layer's state gives a different answer
    only_last = [v.clone() for v in s]
    for v, f in zip(only_last, fin_a):
        v[:] = f[L - 1]
    out_w, _ = _per_layer(cell, layers, x[:, cut:], only_last)
    assert not torch.allclose(out_w, out[:, cut:], rtol=0, atol=1e-6)


def test_layer_states_flag_and_dense_ex_symbols_are_exported_and_declared():
    header = open(os.path.join(ROOT, "include", "ttrnn_b200.h")).read()
    m = re.search(r"#define\s+TTRNN_WS_LAYER_STATES\s+(\d+)", header)
    assert m and int(m.group(1)) == _lib.WS_LAYER_STATES == 2
    assert _lib.WS_LAYER_STATES & _lib.WS_WHOLE_BATCH == 0        # the flags combine
    lib = _lib.load()
    for name in ("ttrnn_dense_rnn_forward_ex", "ttrnn_dense_rnn_backward_ex"):
        assert re.search(r"\b%s\s*\(" % name, header), name
        assert name in _lib.SYMBOLS
        assert getattr(lib, name) is not None
    # the _ex calls are the plain ones plus a trailing int32 flags argument
    assert _lib.SYMBOLS["ttrnn_dense_rnn_forward_ex"][1][:-1] == _lib.SYMBOLS["ttrnn_dense_rnn_forward"][1]
    assert _lib.SYMBOLS["ttrnn_dense_rnn_backward_ex"][1][:-1] == _lib.SYMBOLS["ttrnn_dense_rnn_backward"][1]


def test_module_forward_states_rejects_cpu_tensors():
    """No CPU fallback: the fused path of forward_states raises on CPU tensors like forward() does."""
    import tensorized_rnn_b200 as tr
    with redirect_stdout(io.StringIO()):
        m = tr.TTLSTM(12, 20, 2, torch.device("cpu"), n_cores=2, tt_rank=2)
    with pytest.raises(RuntimeError):
        m.forward_states(torch.rand(2, 3, 12))
