"""References for variable-length rows (DESIGN.md §4.22), test infrastructure only.

`oracle_rows` runs the unchanged oracle row by row on x[b:b+1, :len_b] and pads the outputs with zeros; `torch_packed`
runs torch.nn.LSTM / GRU on a PackedSequence in FP64 with the dense weights formed from the TT cores (oracle.tt_dense).
tests/test_varlen_cpu.py pins the two against each other; the GPU tests compare the engine with both.
"""
import torch
from torch.nn.utils.rnn import pack_padded_sequence, pad_packed_sequence

from helpers import oracle


def oracle_rows(cell, layers, x, lengths, init_states=None):
    """(out (B, T, H) zero past each length, h_n (B, H)[, c_n (B, H)]) of the last layer, the shared-state contract."""
    B, T, _ = x.shape
    outs, hs, cs = [], [], []
    for b, n in enumerate(int(v) for v in lengths):
        xb = x[b:b + 1, :n]
        if cell == "lstm":
            init = None if init_states is None else tuple(s[b:b + 1] for s in init_states)
            o, (h, c) = oracle.lstm_forward(layers, xb, init)
            cs.append(c)
        else:
            init = None if init_states is None else init_states[b:b + 1]
            o, h = oracle.gru_forward(layers, xb, init)
        outs.append(torch.cat([o, o.new_zeros(1, T - n, o.shape[2])], dim=1))
        hs.append(h)
    res = (torch.cat(outs), torch.cat(hs))
    return res + ((torch.cat(cs),) if cell == "lstm" else ())


def torch_module(cell, layers, dtype=torch.float64):
    """torch.nn.LSTM / GRU (batch_first) holding the dense weights of oracle `layers`."""
    first = layers[0]
    W_ih0 = oracle.tt_dense(first["ih_cores"])
    H = oracle.tt_dense(first["hh_cores"]).shape[1]
    bias = first["ih_bias"] is not None
    cls = torch.nn.LSTM if cell == "lstm" else torch.nn.GRU
    m = cls(W_ih0.shape[1], H, len(layers), bias=bias, batch_first=True).to(dtype)
    with torch.no_grad():
        for l, p in enumerate(layers):
            getattr(m, "weight_ih_l%d" % l).copy_(oracle.tt_dense(p["ih_cores"]))
            getattr(m, "weight_hh_l%d" % l).copy_(oracle.tt_dense(p["hh_cores"]))
            if bias:
                getattr(m, "bias_ih_l%d" % l).copy_(p["ih_bias"])
                getattr(m, "bias_hh_l%d" % l).copy_(p["hh_bias"])
    return m


def torch_packed(cell, layers, x, lengths, init_states=None):
    """The same as oracle_rows through torch's PackedSequence path (one shared initial state seeds every layer)."""
    m = torch_module(cell, layers, x.dtype)
    L = len(layers)
    packed = pack_padded_sequence(x, torch.as_tensor(lengths), batch_first=True, enforce_sorted=False)
    if init_states is None:
        hx = None
    elif cell == "lstm":
        hx = tuple(s.unsqueeze(0).expand(L, -1, -1).contiguous() for s in init_states)
    else:
        hx = init_states.unsqueeze(0).expand(L, -1, -1).contiguous()
    out, st = m(packed, hx)
    out, _ = pad_packed_sequence(out, batch_first=True, total_length=x.shape[1])
    if cell == "lstm":
        return out, st[0][-1], st[1][-1]
    return out, st[-1]
