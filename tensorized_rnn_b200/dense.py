"""Dense LSTM / GRU baselines through the same engine (SURVEY.md 8f-3).

Mirrors the reference's `LSTM` / `LSTMCell` (tensorized_rnn/lstm.py:7-41, 44-135) and `GRU` / `GRUCell`
(tensorized_rnn/gru.py:11-50, 52-136): constructor signatures, attribute and sub-module names (`cell{i}.input_weights`,
`cell{i}.hidden_weights` are `nn.Linear`s, so the state_dict keys are `cell{i}.input_weights.weight` ...), the bias
convention (the dense LSTM cell gives its input map NO bias, lstm.py:17-18; the GRU cell gives both maps `bias`,
gru.py:19-23), `init_hidden`, `param_count`, and the forward contract of lstm.py:101-135 / gru.py:104-136.  These are the
modules `pmnist_test.py` builds without `--tt` and `SpeakerEncoder` builds with `compression=None`: with them the
paper's dense-vs-TT comparison runs on the same device path (C ABI `ttrnn_dense_rnn_*`, csrc/tt_dense.cuh).
`bidirectional=True` adds `cell{i}_reverse` per layer and runs the stack as one-layer calls per (layer, direction), as the TT
modules do (functional.bidirectional_stack, DESIGN.md §4.17).
`dropout=p` masks the output of every layer but the last in training mode, as torch.nn.LSTM(dropout=p) does; a stack with
active dropout runs as one-layer calls with the mask kernel between them (DESIGN.md §4.18).
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional

import torch
from torch import nn

from . import _lib
from .functional import _bytes_to_floats, _dense16, _ptr, _require_cuda_f32, bidirectional_stack, layer_dropout, \
    shared_bidirectional_state
from .rnn import active_dropout, check_dropout


class _DenseRnnFunction(torch.autograd.Function):
    """`layer_states`: h0 / c0 and the returned final states are (L, B, H), one block per layer (TTRNN_WS_LAYER_STATES)."""

    @staticmethod
    def forward(ctx, cell: str, hidden_size: int, num_layers: int, has_bias: bool, layer_states: bool, x, h0, c0, *params):
        lib = _lib.load()
        _require_cuda_f32("input", x)
        for i, p in enumerate(params):
            _require_cuda_f32("parameter %d" % i, p)
        if x.dim() != 3:
            raise ValueError("input must be (batch, seq_len, input_size), got shape %s" % (tuple(x.shape),))
        B, T, I = x.shape
        H = hidden_size
        state_shape = (num_layers, B, H) if layer_states else (B, H)
        flags = _lib.WS_LAYER_STATES if layer_states else 0
        for name, s in (("h0", h0), ("c0", c0)):
            if s is not None:
                _require_cuda_f32(name, s)
                if tuple(s.shape) != state_shape:
                    raise ValueError("%s must have shape %s, got %s" % (name, state_shape, tuple(s.shape)))
        x, h0c, c0c = _dense16(x), _dense16(h0), _dense16(c0)
        desc = _lib.DenseDesc(_lib.CELL_LSTM if cell == "lstm" else _lib.CELL_GRU, num_layers, I, H, int(has_bias), T, B)
        with torch.cuda.device(x.device):
            blob = torch.cat([p.detach().reshape(-1) for p in params])
            want = lib.ttrnn_dense_rnn_param_count(C.byref(desc))
            if want < 0:
                raise ValueError("ttrnn_dense_rnn_param_count failed: " + _lib.last_error())
            if want != blob.numel():
                raise RuntimeError("parameter blob has %d floats, descriptor expects %d" % (blob.numel(), want))
            sb, wb = C.c_int64(0), C.c_int64(0)
            _lib.check(lib.ttrnn_dense_rnn_workspace_bytes(C.byref(desc), C.byref(sb), C.byref(wb)), "ttrnn_dense_rnn_workspace_bytes")
            out = torch.empty((B, T, H), device=x.device, dtype=torch.float32)
            hT = torch.empty(state_shape, device=x.device, dtype=torch.float32)
            cT = torch.empty(state_shape, device=x.device, dtype=torch.float32) if cell == "lstm" else None
            saved = torch.empty(_bytes_to_floats(sb.value), device=x.device, dtype=torch.float32)
            scratch = torch.empty(_bytes_to_floats(wb.value), device=x.device, dtype=torch.float32)
            stream = torch.cuda.current_stream(x.device).cuda_stream
            _lib.check(lib.ttrnn_dense_rnn_forward_ex(C.byref(desc), _ptr(x), _ptr(h0c), _ptr(c0c), _ptr(blob), _ptr(out), _ptr(hT),
                                                      _ptr(cT), _ptr(saved), _ptr(scratch), stream, flags), "ttrnn_dense_rnn_forward")
        ctx.desc, ctx.cell = desc, cell
        ctx.flags, ctx.state_shape = flags, state_shape
        ctx.shapes = [tuple(p.shape) for p in params]
        ctx.scratch_floats = _bytes_to_floats(wb.value)
        ctx.has_h0, ctx.has_c0 = h0 is not None, c0 is not None
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(x, h0c, c0c, blob, out, saved)
        return (out, hT, cT) if cell == "lstm" else (out, hT)

    @staticmethod
    def backward(ctx, *grads):
        lib = _lib.load()
        x, h0, c0, blob, out, saved = ctx.saved_tensors
        if getattr(ctx, "consumed", False):
            raise RuntimeError("dense LSTM/GRU: the saved activations were consumed by a previous backward "
                               "(retain_graph is not supported by this path)")
        ctx.consumed = True
        lstm = ctx.cell == "lstm"
        d_out, d_hT = _dense16(grads[0]), _dense16(grads[1])
        d_cT = _dense16(grads[2]) if lstm else None
        B, H = x.shape[0], out.shape[2]
        with torch.cuda.device(x.device):
            d_blob = torch.empty_like(blob)
            d_x = torch.empty_like(x) if ctx.needs_input_grad[5] else None
            d_h0 = torch.empty(ctx.state_shape, device=x.device, dtype=torch.float32) \
                if (ctx.has_h0 and ctx.needs_input_grad[6]) else None
            d_c0 = torch.empty(ctx.state_shape, device=x.device, dtype=torch.float32) \
                if (lstm and ctx.has_c0 and ctx.needs_input_grad[7]) else None
            scratch = torch.empty(ctx.scratch_floats, device=x.device, dtype=torch.float32)
            stream = torch.cuda.current_stream(x.device).cuda_stream
            _lib.check(lib.ttrnn_dense_rnn_backward_ex(C.byref(ctx.desc), _ptr(x), _ptr(h0), _ptr(c0), _ptr(blob), _ptr(out),
                                                       _ptr(saved), _ptr(d_out), _ptr(d_hT), _ptr(d_cT), _ptr(d_blob), _ptr(d_x),
                                                       _ptr(d_h0), _ptr(d_c0), _ptr(scratch), stream, ctx.flags),
                       "ttrnn_dense_rnn_backward")
        d_params, off = [], 0
        for i, shp in enumerate(ctx.shapes):
            n = 1
            for v in shp:
                n *= v
            d_params.append(d_blob[off:off + n].view(shp) if ctx.needs_input_grad[8 + i] else None)
            off += n
        return (None, None, None, None, None, d_x, d_h0, d_c0) + tuple(d_params)


class _DenseCell(nn.Module):
    n_gate = 0

    def __init__(self, input_size, hidden_size, bias, device):
        super().__init__()
        self.input_size, self.hidden_size, self.bias, self.device = input_size, hidden_size, bias, device
        self.input_weights = self._create_input_hidden_weights()
        self.hidden_weights = self._create_hidden_hidden_weights()

    def flat_parameters(self) -> List[torch.Tensor]:
        out = [self.input_weights.weight]
        if self.input_weights.bias is not None:
            out.append(self.input_weights.bias)
        out.append(self.hidden_weights.weight)
        if self.hidden_weights.bias is not None:
            out.append(self.hidden_weights.bias)
        return out


class LSTMCell(_DenseCell):
    """Weights of one dense LSTM layer (reference lstm.py:7-21).  The step itself runs inside the sequence call."""
    n_gate = 4

    def _create_input_hidden_weights(self):
        return nn.Linear(self.input_size, 4 * self.hidden_size, False).to(self.device)      # lstm.py:18: no bias

    def _create_hidden_hidden_weights(self):
        return nn.Linear(self.hidden_size, 4 * self.hidden_size, self.bias).to(self.device)


class GRUCell(_DenseCell):
    """Weights of one dense GRU layer (reference gru.py:11-23)."""
    n_gate = 3

    def _create_input_hidden_weights(self):
        return nn.Linear(self.input_size, 3 * self.hidden_size, self.bias).to(self.device)

    def _create_hidden_hidden_weights(self):
        return nn.Linear(self.hidden_size, 3 * self.hidden_size, self.bias).to(self.device)


class _DenseRnnBase(nn.Module):
    cell_kind = ""
    cell_cls = None

    def __init__(self, input_size, hidden_size, num_layers, device, bias=True, log_grads=False, bidirectional=False,
                 dropout=0.0):
        dropout = check_dropout(dropout, num_layers)
        super().__init__()
        self.input_size, self.hidden_size, self.num_layers = input_size, hidden_size, num_layers
        self.bias, self.device, self.log_grads = bias, device, log_grads
        self.bidirectional = bool(bidirectional)
        self.dropout = dropout
        if log_grads:
            raise NotImplementedError("log_grads=True is implemented for the TT modules (TTLSTM / TTGRU); the dense baselines "
                                      "run as one fused sequence call and expose no per-step hooks")
        # bidirectional: cell{i}_reverse after cell{i}, and the layers above the first take both directions' outputs
        self._all_layers = []
        for i in range(num_layers):
            in_size = input_size if i == 0 else (2 * hidden_size if self.bidirectional else hidden_size)
            for name in ("cell{}", "cell{}_reverse") if self.bidirectional else ("cell{}",):
                cell = self.cell_cls(in_size, hidden_size, bias, device)
                setattr(self, name.format(i), cell)
                self._all_layers.append(cell)

    def param_count(self):
        return int(sum(p.numel() for c in self._all_layers for p in c.parameters()))

    def flat_parameters(self):
        return [p for c in self._all_layers for p in c.flat_parameters()]

    def _run(self, input, h0, c0, layer_states=False):
        if input.shape[1] == 0:
            raise NameError("name 'x' is not defined")       # the reference fails the same way on T = 0 (lstm.py:135)
        if self.bidirectional:
            return self._run_bidirectional(input, h0, c0, layer_states)
        dropout = active_dropout(self, input.device)
        if dropout is not None:
            return self._run_layers(input, h0, c0, layer_states, dropout)
        return _DenseRnnFunction.apply(self.cell_kind, self.hidden_size, self.num_layers, bool(self.bias), layer_states, input,
                                       h0, c0, *self.flat_parameters())

    def _run_layers(self, input, h0, c0, layer_states, dropout):
        """A unidirectional stack with inter-layer dropout: one one-layer sequence call per layer, the mask kernel between
        them (functional.layer_dropout).  layer_states: h0 / c0 (L, B, H), every layer's final states returned; else one
        (B, H) state seeds every layer and the last layer's final states come back."""
        states = [h0, c0] if self.cell_kind == "lstm" else [h0]
        shape = (self.num_layers, input.size(0), self.hidden_size)
        if layer_states:
            for s in states:
                if s is not None and tuple(s.shape) != shape:
                    raise ValueError("per-layer states must have shape %s, got %s" % (shape, tuple(s.shape)))
        inp, fins = input, []
        for l, cell in enumerate(self._all_layers):
            st = [None if s is None else (s[l] if layer_states else s) for s in states]
            res = _DenseRnnFunction.apply(self.cell_kind, self.hidden_size, 1, bool(self.bias), False, inp, *st,
                                          *([None] if self.cell_kind == "gru" else []), *cell.flat_parameters())
            inp = res[0] if l == self.num_layers - 1 else layer_dropout(res[0], dropout, l)
            fins.append(res[1:])
        if layer_states:
            return (inp, *[torch.stack([f[k] for f in fins]) for k in range(len(states))])
        return (inp, *fins[-1])

    def _run_bidirectional(self, input, h0, c0, layer_states):
        """Every (layer, direction) is a one-layer sequence call (functional.bidirectional_stack).  layer_states: h0 / c0
        are (2L, B, H) and so are the returned final states; else one (B, H) state seeds every layer and both directions
        and the last layer's two directions' final states come back as (2, B, H)."""
        def run(layer, direction, x, h, c=None):
            cell = self._all_layers[2 * layer + direction]
            return _DenseRnnFunction.apply(self.cell_kind, self.hidden_size, 1, bool(self.bias), False, x, h, c,
                                           *cell.flat_parameters())

        states = [h0, c0] if self.cell_kind == "lstm" else [h0]
        if not layer_states:
            states = [shared_bidirectional_state(s, self.num_layers, input.size(0), self.hidden_size) for s in states]
        out, fin = bidirectional_stack(input, states, self.num_layers, self.hidden_size, run,
                                       dropout=active_dropout(self, input.device))
        if not layer_states:
            fin = [f[-2:] for f in fin]
        return (out, *fin)


class LSTM(_DenseRnnBase):
    """Dense LSTM stack, drop-in for reference tensorized_rnn.lstm.LSTM (lstm.py:44-135)."""
    cell_kind, cell_cls = "lstm", LSTMCell

    def init_hidden(self, batch_size):
        h = torch.zeros(batch_size, self.hidden_size).to(self.device)
        return h, torch.zeros(batch_size, self.hidden_size).to(self.device)

    def forward(self, input, init_states=None):
        h0, c0 = init_states if init_states is not None else (None, None)
        out, h, c = self._run(input, h0, c0)
        return out, (h, c)

    def forward_states(self, input, states=None):
        """Per-layer states, as torch.nn.LSTM takes them: `states` = (h, c), each (num_layers, batch, hidden), or None
        (zeros).  Returns (outputs, (h_n, c_n)) with every layer's final state, so a sequence can be run in pieces."""
        h0, c0 = states if states is not None else (None, None)
        out, h, c = self._run(input, h0, c0, layer_states=True)
        return out, (h, c)


class GRU(_DenseRnnBase):
    """Dense GRU stack, drop-in for reference tensorized_rnn.gru.GRU (gru.py:52-136)."""
    cell_kind, cell_cls = "gru", GRUCell

    def init_hidden(self, batch_size):
        return torch.zeros(batch_size, self.hidden_size).to(self.device)

    def forward(self, input, init_states=None):
        out, h = self._run(input, init_states, None)
        return out, h

    def forward_states(self, input, states=None):
        """Per-layer states: `states` (num_layers, batch, hidden) or None (zeros) -> (outputs, h_n (num_layers, batch,
        hidden))."""
        return self._run(input, states, None, layer_states=True)
