"""autograd glue between the nn.Module mirror and the C ABI.

One `torch.autograd.Function` per whole-sequence call: forward packs every core and bias into one
contiguous FP32 blob (the layout of include/ttrnn_b200.h), lets torch own every buffer, and calls
`ttrnn_rnn_forward`; backward calls `ttrnn_rnn_backward` and hands each parameter its slice of the
gradient blob.  PyTorch is plumbing here (memory, streams, autograd bookkeeping); all arithmetic of
the path runs in the CUDA library.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _require_cuda_f32(name: str, t: torch.Tensor) -> None:
    if not t.is_cuda:
        raise RuntimeError("tensorized_rnn_b200: `%s` is on %s; the engine runs on CUDA (sm_100a) only and has "
                           "no CPU fallback" % (name, t.device))
    if t.dtype != torch.float32:
        raise TypeError("tensorized_rnn_b200: `%s` must be float32 (the path is FP32 end to end), got %s"
                        % (name, t.dtype))


class RnnSpec(object):
    """Static description of a TT-RNN stack: cell kind, sizes and the TT shape of every weight.  `proj_size` > 0 (LSTM
    only) with `hr_shapes`: the projected LSTM, whose layers output h_t = W_hr m_t of width proj_size (DESIGN.md §4.19)."""

    def __init__(self, cell: str, input_size: int, hidden_size: int, has_bias: bool,
                 ih_shapes: Sequence[Tuple[Sequence[int], Sequence[int], Sequence[int]]],
                 hh_shapes: Sequence[Tuple[Sequence[int], Sequence[int], Sequence[int]]],
                 proj_size: int = 0,
                 hr_shapes: Optional[Sequence[Tuple[Sequence[int], Sequence[int], Sequence[int]]]] = None):
        assert cell in ("lstm", "gru")
        self.cell = cell
        self.n_gates = 4 if cell == "lstm" else 3
        self.input_size, self.hidden_size, self.has_bias = int(input_size), int(hidden_size), bool(has_bias)
        self.num_layers = len(ih_shapes)
        if self.num_layers > _lib.MAX_LAYERS:
            raise ValueError("at most %d layers are supported" % _lib.MAX_LAYERS)
        self.ih_shapes = [tuple(list(map(int, v)) for v in s) for s in ih_shapes]   # (in_modes, out_modes, ranks)
        self.hh_shapes = [tuple(list(map(int, v)) for v in s) for s in hh_shapes]
        self.proj_size = int(proj_size)
        self.hr_shapes = [tuple(list(map(int, v)) for v in s) for s in hr_shapes] if self.proj_size else []
        assert not self.proj_size or (cell == "lstm" and len(self.hr_shapes) == self.num_layers)
        self.output_size = self.proj_size or self.hidden_size       # width of h_t and of every layer's output
        self._proj = None
        self._cache = {}

    def proj(self) -> Optional[_lib.RnnProj]:
        """The ttrnn_rnn_proj of a projected stack, else None."""
        if not self.proj_size:
            return None
        if self._proj is None:
            pj = _lib.RnnProj()
            pj.proj_size, pj.reserved = self.proj_size, 0
            for l in range(self.num_layers):
                pj.hr[l] = _lib.make_tt_shape(*self.hr_shapes[l])
            self._proj = pj
        return self._proj

    def desc(self, batch: int, seq_len: int) -> _lib.RnnDesc:
        key = (batch, seq_len)
        d = self._cache.get(key)
        if d is None:
            d = _lib.RnnDesc()
            d.cell = _lib.CELL_LSTM if self.cell == "lstm" else _lib.CELL_GRU
            d.num_layers, d.input_size, d.hidden_size = self.num_layers, self.input_size, self.hidden_size
            d.has_bias, d.seq_len, d.batch = int(self.has_bias), seq_len, batch
            for l in range(self.num_layers):
                d.ih[l] = _lib.make_tt_shape(*self.ih_shapes[l])
                d.hh[l] = _lib.make_tt_shape(*self.hh_shapes[l])
            if len(self._cache) > 64:
                self._cache.clear()
            self._cache[key] = d
        return d


def _bytes_to_floats(nbytes: int) -> int:
    return max(1, (int(nbytes) + 3) // 4)


def _dense16(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    """Contiguous and 16-byte aligned: the kernels read these buffers with float4 loads, 16-byte cp.async and TMA.
    `.contiguous()` keeps a contiguous view whose storage offset is not a multiple of 4 floats (a slice of a flat
    buffer); such a view is copied."""
    if t is None:
        return None
    t = t.contiguous()
    if t.data_ptr() % 16 != 0:
        t = t.clone()
    return t


def _step_stats(lib, v: torch.Tensor, stream) -> torch.Tensor:
    """(2, T): mean_b ||v[b,t]||^2 and mean_b log ||v[b,t]||^2 of a contiguous (B,T,H) block (ttrnn_step_norms)."""
    B, T, H = v.shape
    out = torch.empty((2, T), device=v.device, dtype=torch.float32)
    _lib.check(lib.ttrnn_step_norms(_ptr(v), B, T, H, _ptr(out), stream), "ttrnn_step_norms")
    return out


def dropout_draw(device: torch.device) -> Tuple[int, int]:
    """(seed, offset) of one dropout mask from the device's default CUDA generator, which advances by 4 per draw: so
    torch.manual_seed / torch.cuda.manual_seed reproduce a run and two successive calls draw different masks.  The
    generator's offset is host state that a replayed CUDA graph would not advance, so drawing under stream capture is an
    error."""
    if torch.cuda.is_current_stream_capturing():
        raise RuntimeError("tensorized_rnn_b200: dropout draws its mask offset from the CUDA generator on the host, which "
                           "is not graph-safe; capture the module in eval mode or with dropout=0")
    idx = device.index if device.index is not None else torch.cuda.current_device()
    gen = torch.cuda.default_generators[idx]
    seed, offset = int(gen.initial_seed()), int(gen.get_offset())
    gen.set_offset(offset + 4)
    return seed, offset


def _dropout_struct(dropout) -> _lib.Dropout:
    p, seed, offset = dropout
    d = _lib.Dropout()
    d.p, d.reserved, d.seed, d.offset = float(p), 0, int(seed) & (2 ** 64 - 1), int(offset) & (2 ** 64 - 1)
    return d


class _DropoutFunction(torch.autograd.Function):
    """y = x * mask / (1 - p) of one layer boundary (ttrnn_dropout_apply), `dropout` = (p, seed, offset).  With `rev`
    also y reversed in time (the next bidirectional layer's reverse-direction input); the backward forms
    d_x = (dy + reverse(dy_rev)) * mask / (1 - p) in the same kernel, regenerating the mask."""

    @staticmethod
    def forward(ctx, dropout, boundary: int, rev: bool, x):
        lib = _lib.load()
        _require_cuda_f32("input", x)
        x = _dense16(x)
        B, T, F = x.shape
        dp = _dropout_struct(dropout)
        with torch.cuda.device(x.device):
            y = torch.empty_like(x)
            y_rev = torch.empty_like(x) if rev else None
            _lib.check(lib.ttrnn_dropout_apply(B, T, F, 0, boundary, 0, C.byref(dp), _ptr(x), _ptr(y), _ptr(y_rev),
                                               torch.cuda.current_stream(x.device).cuda_stream), "ttrnn_dropout_apply")
        ctx.dropout, ctx.boundary = dropout, boundary
        ctx.set_materialize_grads(False)
        return (y, y_rev) if rev else y

    @staticmethod
    def backward(ctx, dy, dy_rev=None):
        if dy is None and dy_rev is None:
            return None, None, None, None
        lib = _lib.load()
        dy, dy_rev = _dense16(dy), _dense16(dy_rev)
        like = dy if dy is not None else dy_rev
        B, T, F = like.shape
        dp = _dropout_struct(ctx.dropout)
        with torch.cuda.device(like.device):
            d_x = torch.empty_like(like)
            src = dy if dy is not None else torch.zeros_like(like)
            _lib.check(lib.ttrnn_dropout_apply(B, T, F, 0, ctx.boundary, 1, C.byref(dp), _ptr(src), _ptr(d_x), _ptr(dy_rev),
                                               torch.cuda.current_stream(like.device).cuda_stream), "ttrnn_dropout_apply")
        return None, None, None, d_x


def layer_dropout(x: torch.Tensor, dropout, boundary: int, rev: bool = False):
    """The inter-layer dropout of a stack composed of one-layer calls: the output x (B, T, F) of layer `boundary` times
    mask / (1 - p), the mask drawn from `dropout` = (p, seed, offset) as the whole-stack call draws it (DESIGN.md
    §4.18).  rev: returns (y, y reversed in time)."""
    return _DropoutFunction.apply(dropout, int(boundary), bool(rev), x)


def check_lengths(lengths, batch: int, seq_len: int, device: torch.device) -> torch.Tensor:
    """Per-row lengths of a padded (batch, seq_len, .) input as the int32 device array the _lengths entry points take.
    Checked on the host before the copy (1 <= len_b <= seq_len): the kernels trust them (DESIGN.md §4.22)."""
    host = torch.as_tensor(lengths).detach().to("cpu")
    if host.dtype.is_floating_point or host.dtype == torch.bool or host.dim() != 1 or host.numel() != batch:
        raise ValueError("lengths must be %d integers (one per batch row), got %s of shape %s"
                         % (batch, host.dtype, tuple(host.shape)))
    if host.numel() and (int(host.min()) < 1 or int(host.max()) > seq_len):
        raise ValueError("lengths must be in [1, %d] (the padded sequence length), got min %d, max %d"
                         % (seq_len, int(host.min()), int(host.max())))
    return host.to(torch.int32).to(device)


def unpack_sequence(packed):
    """A torch PackedSequence as (padded (B, T, F) zero-padded in the caller's batch order, lengths (B,) on the host)."""
    return torch.nn.utils.rnn.pad_packed_sequence(packed, batch_first=True, padding_value=0.0)


def pack_like(padded: torch.Tensor, lengths: torch.Tensor, like) -> "torch.nn.utils.rnn.PackedSequence":
    """The (B, T, .) output of a padded run as a PackedSequence with the batch_sizes, sorted_indices and unsorted_indices
    of the input `like` (rows are put in like's sorted order first, so that ties keep its order)."""
    idx = like.sorted_indices
    if idx is not None:
        padded, lengths = padded.index_select(0, idx), lengths.index_select(0, idx.to(lengths.device))
    data = torch.nn.utils.rnn.pack_padded_sequence(padded, lengths, batch_first=True, enforce_sorted=True).data
    return torch.nn.utils.rnn.PackedSequence(data, like.batch_sizes, like.sorted_indices, like.unsorted_indices)


class _RnnFunction(torch.autograd.Function):
    """`step_log` (None or an object with .activations(layer, var, stats) / .gradients(layer, var, stats)): fused
    log_grads.  The training forward reports the per-step statistics of every layer's h_t / c_t sequence, the
    backward those of the total gradients reaching them, (2, T) tensors each (reference rnn_utils.py:127-172).
    `layer_states`: h0 / c0 and the returned final states are (L, B, H), one block per layer (TTRNN_WS_LAYER_STATES);
    else (B, H), shared by every layer on the way in and the last layer's on the way out.
    `dropout`: None, or (p, seed, offset) of the inter-layer dropout (ttrnn_rnn_forward_dropout, TTRNN_WS_DROPOUT); the
    backward regenerates the same mask from them.
    A projected spec (proj_size P > 0) runs the _proj entry points: out and the h states are P wide, the c states H.
    `lengths`: None, or the int32 device array of per-row lengths (check_lengths): the _lengths entry points."""

    @staticmethod
    def forward(ctx, spec: RnnSpec, grad_enabled: bool, step_log, layer_states: bool, dropout, lengths, x, h0, c0, *params):
        lib = _lib.load()
        _require_cuda_f32("input", x)
        for i, p in enumerate(params):
            _require_cuda_f32("parameter %d" % i, p)
            if p.device != x.device:
                raise RuntimeError("parameter %d is on %s but the input is on %s" % (i, p.device, x.device))
        B, T, I = x.shape
        H, W = spec.hidden_size, spec.output_size
        if I != spec.input_size:
            raise ValueError("input has %d features, the module was built for %d" % (I, spec.input_size))
        lead = (spec.num_layers, B) if layer_states else (B,)
        state_shape, h_shape = lead + (H,), lead + (W,)
        for name, s, shp in (("h0", h0, h_shape), ("c0", c0, state_shape)):
            if s is not None:
                _require_cuda_f32(name, s)
                if tuple(s.shape) != shp:
                    raise ValueError("%s must have shape %s, got %s" % (name, shp, tuple(s.shape)))
        x = _dense16(x)
        h0c = _dense16(h0)
        c0c = _dense16(c0)
        desc = spec.desc(B, T)
        with torch.cuda.device(x.device):
            blob = torch.cat([p.detach().reshape(-1) for p in params])
            pj = spec.proj()
            want = lib.ttrnn_rnn_param_count(C.byref(desc)) if pj is None else \
                lib.ttrnn_rnn_param_count_proj(C.byref(desc), C.byref(pj))
            if want < 0:
                raise RuntimeError("ttrnn_rnn_param_count failed: " + _lib.last_error())
            if want != blob.numel():
                raise RuntimeError("parameter blob has %d floats, descriptor expects %d" % (blob.numel(), want))
            ws = _lib.RnnWorkspace()
            flags = (_lib.WS_WHOLE_BATCH if step_log is not None else 0) | (_lib.WS_LAYER_STATES if layer_states else 0) | \
                (_lib.WS_DROPOUT if dropout is not None else 0) | (_lib.WS_LENGTHS if lengths is not None else 0)
            if pj is None:
                _lib.check(lib.ttrnn_rnn_workspace_bytes_ex(C.byref(desc), flags, C.byref(ws)), "ttrnn_rnn_workspace_bytes")
            else:
                _lib.check(lib.ttrnn_rnn_workspace_bytes_proj(C.byref(desc), C.byref(pj), flags | _lib.WS_PROJ, C.byref(ws)),
                           "ttrnn_rnn_workspace_bytes_proj")
            # grad mode is always off inside Function.forward and needs_input_grad stays True for nn.Parameters under
            # torch.no_grad(): the caller captures torch.is_grad_enabled() before .apply (ADVICE r1)
            training = bool(grad_enabled) and any(ctx.needs_input_grad[6:])
            if step_log is not None and not training:
                raise RuntimeError("fused per-step logging needs a training forward (it reads the kept h_t / c_t sequences)")
            out = torch.empty((B, T, W), device=x.device, dtype=torch.float32)
            hT = torch.empty(h_shape, device=x.device, dtype=torch.float32)
            cT = torch.empty(state_shape, device=x.device, dtype=torch.float32) if spec.cell == "lstm" else None
            saved = torch.empty(_bytes_to_floats(ws.saved_bytes), device=x.device, dtype=torch.float32) \
                if training else None
            scratch = torch.empty(_bytes_to_floats(ws.fwd_scratch_bytes), device=x.device, dtype=torch.float32)
            stream = torch.cuda.current_stream(x.device).cuda_stream
            args = (C.byref(desc), C.byref(ws), _ptr(x), _ptr(h0c), _ptr(c0c), _ptr(blob), _ptr(out), _ptr(hT), _ptr(cT),
                    _ptr(saved), _ptr(scratch), stream)
            if lengths is not None:
                dp = None if dropout is None else C.byref(_dropout_struct(dropout))
                _lib.check(lib.ttrnn_rnn_forward_lengths(*(args + (None if pj is None else C.byref(pj), dp, _ptr(lengths)))),
                           "ttrnn_rnn_forward_lengths")
            elif pj is not None:
                dp = None if dropout is None else C.byref(_dropout_struct(dropout))
                _lib.check(lib.ttrnn_rnn_forward_proj(*(args + (C.byref(pj), dp))), "ttrnn_rnn_forward_proj")
            elif dropout is None:
                _lib.check(lib.ttrnn_rnn_forward(*args), "ttrnn_rnn_forward")
            else:
                _lib.check(lib.ttrnn_rnn_forward_dropout(*(args + (C.byref(_dropout_struct(dropout)),))),
                           "ttrnn_rnn_forward_dropout")
            if step_log is not None:
                hs_off, cs_off = C.c_int64(), C.c_int64()
                for l in range(spec.num_layers):
                    _lib.check(lib.ttrnn_rnn_saved_layout(C.byref(desc), C.byref(ws), l, C.byref(hs_off), C.byref(cs_off)),
                               "ttrnn_rnn_saved_layout")
                    hs = out if hs_off.value < 0 else saved[hs_off.value:hs_off.value + B * T * H].view(B, T, H)
                    step_log.activations(l, "h", _step_stats(lib, hs, stream))
                    if cs_off.value >= 0:
                        step_log.activations(l, "c", _step_stats(lib, saved[cs_off.value:cs_off.value + B * T * H].view(B, T, H), stream))
        if training:
            ctx.spec = spec
            ctx.step_log = step_log
            ctx.dropout = dropout
            ctx.lengths = lengths
            ctx.shapes = [tuple(p.shape) for p in params]
            ctx.ws = ws                    # sizes + execution plan: backward runs from the same plan as this forward
            ctx.bwd_floats = _bytes_to_floats(ws.bwd_scratch_bytes)
            ctx.has_h0, ctx.has_c0 = h0 is not None, c0 is not None
            ctx.state_shape, ctx.h_shape = state_shape, h_shape
            ctx.set_materialize_grads(False)
            ctx.save_for_backward(x, h0c, c0c, blob, out, saved)
        if spec.cell == "lstm":
            return out, hT, cT
        return out, hT

    @staticmethod
    def backward(ctx, *grads):
        lib = _lib.load()
        spec: RnnSpec = ctx.spec
        x, h0, c0, blob, out, saved = ctx.saved_tensors
        d_out = grads[0]
        d_hT = grads[1]
        d_cT = grads[2] if spec.cell == "lstm" else None
        B, T, _ = x.shape
        H = spec.hidden_size
        desc = spec.desc(B, T)
        d_out = _dense16(d_out)            # the BPTT kernels stage dOut tiles with 16-byte cp.async
        d_hT = _dense16(d_hT)
        d_cT = _dense16(d_cT)
        with torch.cuda.device(x.device):
            d_blob = torch.empty_like(blob)
            d_x = torch.empty_like(x) if ctx.needs_input_grad[6] else None
            d_h0 = torch.empty(ctx.h_shape, device=x.device, dtype=torch.float32) \
                if (ctx.has_h0 and ctx.needs_input_grad[7]) else None
            d_c0 = torch.empty(ctx.state_shape, device=x.device, dtype=torch.float32) \
                if (spec.cell == "lstm" and ctx.has_c0 and ctx.needs_input_grad[8]) else None
            scratch = torch.empty(ctx.bwd_floats, device=x.device, dtype=torch.float32)
            stream = torch.cuda.current_stream(x.device).cuda_stream
            args = (C.byref(desc), C.byref(ctx.ws), _ptr(x), _ptr(h0), _ptr(c0), _ptr(blob), _ptr(out),
                    _ptr(saved), _ptr(d_out), _ptr(d_hT), _ptr(d_cT), _ptr(d_blob),
                    _ptr(d_x), _ptr(d_h0), _ptr(d_c0), _ptr(scratch), stream)
            if ctx.lengths is not None:
                dp = None if ctx.dropout is None else C.byref(_dropout_struct(ctx.dropout))
                pj = C.byref(spec.proj()) if spec.proj_size else None
                _lib.check(lib.ttrnn_rnn_backward_lengths(*(args + (pj, dp, _ptr(ctx.lengths)))), "ttrnn_rnn_backward_lengths")
            elif spec.proj_size:
                dp = None if ctx.dropout is None else C.byref(_dropout_struct(ctx.dropout))
                _lib.check(lib.ttrnn_rnn_backward_proj(*(args + (C.byref(spec.proj()), dp))), "ttrnn_rnn_backward_proj")
            elif ctx.dropout is not None:
                _lib.check(lib.ttrnn_rnn_backward_dropout(*(args + (C.byref(_dropout_struct(ctx.dropout)),))),
                           "ttrnn_rnn_backward_dropout")
            elif ctx.step_log is None:
                _lib.check(lib.ttrnn_rnn_backward(*args), "ttrnn_rnn_backward")
            else:
                L = spec.num_layers
                dh_log = torch.empty((L, B, T, H), device=x.device, dtype=torch.float32)
                dc_log = torch.empty((L, B, T, H), device=x.device, dtype=torch.float32) if spec.cell == "lstm" else None
                _lib.check(lib.ttrnn_rnn_backward_logged(*(args + (_ptr(dh_log), _ptr(dc_log)))), "ttrnn_rnn_backward_logged")
                for l in range(L):
                    ctx.step_log.gradients(l, "h", _step_stats(lib, dh_log[l], stream))
                    if dc_log is not None:
                        ctx.step_log.gradients(l, "c", _step_stats(lib, dc_log[l], stream))
        d_params: List[Optional[torch.Tensor]] = []
        off = 0
        for i, shp in enumerate(ctx.shapes):
            n = 1
            for v in shp:
                n *= v
            d_params.append(d_blob[off:off + n].view(shp) if ctx.needs_input_grad[9 + i] else None)
            off += n
        return (None, None, None, None, None, None, d_x, d_h0, d_c0) + tuple(d_params)


def rnn_sequence(spec: RnnSpec, x: torch.Tensor, h0: Optional[torch.Tensor], c0: Optional[torch.Tensor],
                 params: Sequence[torch.Tensor], step_log=None, layer_states: bool = False, dropout=None, lengths=None):
    """Run the whole stack over the whole sequence.  Returns (out, hT[, cT]).  `step_log`: see _RnnFunction.
    `layer_states=True`: h0 / c0 and the returned hT / cT are (num_layers, batch, hidden), one state per layer, so that
    the final states of one call can seed the next call over the rest of the sequence.
    `dropout`: None, or (p, seed, offset) (dropout_draw): the output of every layer but the last is multiplied by
    mask / (1 - p) before the next layer reads it (DESIGN.md §4.18).
    `lengths`: None, or one length per batch row (1 <= len_b <= seq_len; a sequence or a tensor, checked on the host):
    the padded form of torch's PackedSequence (DESIGN.md §4.22).  Row b runs len_b steps; out is 0 past
    them, hT / cT are the states after step len_b - 1, and the output gradient past them is ignored.  Padded inputs
    must be finite."""
    if x.dim() != 3:
        raise ValueError("input must be (batch, seq_len, input_size), got shape %s" % (tuple(x.shape),))
    if dropout is not None and step_log is not None:
        raise NotImplementedError("inter-layer dropout has no fused per-step logging form")
    if lengths is not None:
        if step_log is not None:
            raise NotImplementedError("variable-length rows have no fused per-step logging form")
        lengths = check_lengths(lengths, x.shape[0], x.shape[1], x.device)
    return _RnnFunction.apply(spec, torch.is_grad_enabled(), step_log, bool(layer_states), dropout, lengths, x, h0, c0,
                              *params)


# ---- bidirectional stacks (DESIGN.md §4.17) --------------------------------------------------------------------------
class _BidirInputFunction(torch.autograd.Function):
    """Layer-0 input of a bidirectional stack: x for the forward direction, x reversed in time for the reverse one
    (ttrnn_time_reverse_add with a = NULL).  The backward forms d_x = d_x_forward + reverse(d_x_reverse) in the same
    kernel, so the two directions' input gradients are summed by the library, not by autograd.
    `lengths` (check_lengths' device array or None): every row is reversed over its own length and zero past it
    (ttrnn_time_reverse_add_lengths)."""

    @staticmethod
    def _reverse_add(lengths, B, T, F, a, r, y, stream):
        lib = _lib.load()
        if lengths is None:
            _lib.check(lib.ttrnn_time_reverse_add(B, T, F, _ptr(a), _ptr(r), _ptr(y), stream), "ttrnn_time_reverse_add")
        else:
            _lib.check(lib.ttrnn_time_reverse_add_lengths(B, T, F, _ptr(a), _ptr(r), _ptr(y), _ptr(lengths), stream),
                       "ttrnn_time_reverse_add_lengths")

    @staticmethod
    def forward(ctx, lengths, x):
        _require_cuda_f32("input", x)
        B, T, F = x.shape
        x = _dense16(x)
        with torch.cuda.device(x.device):
            x_rev = torch.empty_like(x)
            _BidirInputFunction._reverse_add(lengths, B, T, F, None, x, x_rev, torch.cuda.current_stream(x.device).cuda_stream)
        ctx.lengths = lengths
        ctx.set_materialize_grads(False)
        return x, x_rev

    @staticmethod
    def backward(ctx, d_x_f, d_x_r):
        if d_x_f is None and d_x_r is None:
            return None, None
        d_x_f, d_x_r = _dense16(d_x_f), _dense16(d_x_r)
        like = d_x_f if d_x_f is not None else d_x_r
        B, T, F = like.shape
        with torch.cuda.device(like.device):
            d_x = torch.empty_like(like)
            _BidirInputFunction._reverse_add(ctx.lengths, B, T, F, d_x_f, d_x_r, d_x,
                                             torch.cuda.current_stream(like.device).cuda_stream)
        return None, d_x


class _ReverseFunction(torch.autograd.Function):
    """y reversed in time over each row's length (zero past it); its adjoint is the same reversal."""

    @staticmethod
    def forward(ctx, lengths, y):
        y = _dense16(y)
        B, T, F = y.shape
        with torch.cuda.device(y.device):
            y_rev = torch.empty_like(y)
            _BidirInputFunction._reverse_add(lengths, B, T, F, None, y, y_rev, torch.cuda.current_stream(y.device).cuda_stream)
        ctx.lengths = lengths
        return y_rev

    @staticmethod
    def backward(ctx, d_rev):
        d_rev = _dense16(d_rev)
        B, T, F = d_rev.shape
        with torch.cuda.device(d_rev.device):
            d_y = torch.empty_like(d_rev)
            _BidirInputFunction._reverse_add(ctx.lengths, B, T, F, None, d_rev, d_y,
                                             torch.cuda.current_stream(d_rev.device).cuda_stream)
        return None, d_y


class _BidirJoinFunction(torch.autograd.Function):
    """Joins the two directions of one layer (ttrnn_bidir_join): y[b,t] = [out_f[b,t] | out_r[b,T-1-t]], the next
    layer's (or the module's) output, and unless `last`, y reversed in time, the next layer's reverse-direction input.
    `lengths` (device array or None): reversal over each row's length, zeros past it (ttrnn_bidir_join_lengths)."""

    @staticmethod
    def _join(lengths, B, T, H, backward, p, q, u, v, stream):
        lib = _lib.load()
        if lengths is None:
            _lib.check(lib.ttrnn_bidir_join(B, T, H, backward, _ptr(p), _ptr(q), _ptr(u), _ptr(v), stream), "ttrnn_bidir_join")
        else:
            _lib.check(lib.ttrnn_bidir_join_lengths(B, T, H, backward, _ptr(p), _ptr(q), _ptr(u), _ptr(v), _ptr(lengths),
                                                    stream), "ttrnn_bidir_join_lengths")

    @staticmethod
    def forward(ctx, last: bool, lengths, out_f, out_r):
        out_f, out_r = _dense16(out_f), _dense16(out_r)
        B, T, H = out_f.shape
        with torch.cuda.device(out_f.device):
            y = torch.empty((B, T, 2 * H), device=out_f.device, dtype=torch.float32)
            y_rev = None if last else torch.empty_like(y)
            _BidirJoinFunction._join(lengths, B, T, H, 0, out_f, out_r, y, y_rev,
                                     torch.cuda.current_stream(out_f.device).cuda_stream)
        ctx.lengths = lengths
        ctx.set_materialize_grads(False)
        return y if last else (y, y_rev)

    @staticmethod
    def backward(ctx, dy, dy_rev=None):
        if dy is None and dy_rev is None:
            return None, None, None, None
        dy, dy_rev = _dense16(dy), _dense16(dy_rev)
        like = dy if dy is not None else dy_rev
        B, T, H2 = like.shape
        with torch.cuda.device(like.device):
            d_f = torch.empty((B, T, H2 // 2), device=like.device, dtype=torch.float32)
            d_r = torch.empty_like(d_f)
            _BidirJoinFunction._join(ctx.lengths, B, T, H2 // 2, 1, dy, dy_rev, d_f, d_r,
                                     torch.cuda.current_stream(like.device).cuda_stream)
        return None, None, d_f, d_r


_side_streams = {}


def _side_stream(device: torch.device) -> torch.cuda.Stream:
    """The stream the reverse directions run on: one per device, created on first use."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    s = _side_streams.get(idx)
    if s is None:
        s = _side_streams[idx] = torch.cuda.Stream(device=idx)
    return s


def shared_bidirectional_state(state: Optional[torch.Tensor], num_layers: int, batch: int, width: int):
    """forward()'s one (B, width) initial state, which seeds every layer and both directions, as (2L, B, width) views of
    it.  width: the size of that state variable (the hidden size; the projection size for a projected LSTM's h)."""
    if state is None:
        return None
    if tuple(state.shape) != (batch, width):
        raise ValueError("init_states must have shape %s, got %s" % ((batch, width), tuple(state.shape)))
    return state.unsqueeze(0).expand(2 * num_layers, batch, width)


def bidirectional_stack(x: torch.Tensor, states: Sequence[Optional[torch.Tensor]], num_layers: int, hidden_size: int,
                        run, dropout=None, output_size: Optional[int] = None, lengths=None):
    """A bidirectional stack composed of one-layer calls, the contract of torch.nn.LSTM / GRU(bidirectional=True).

    `run(layer, direction, x, *states)` runs direction 0 (forward) or 1 (reverse) of one layer over x (B, T, F) from its
    initial states (None = zeros) with the existing one-layer call and returns (out (B, T, W), *final states).
    W = output_size (the projection size of a projected LSTM), default hidden_size: the width of the output and of the
    h state; every other state (c) is hidden_size wide.
    `states`: one entry per state variable (h, and c for an LSTM), each (2L, B, width) with direction d of layer l at
    2l + d, or None (zeros).  Returns (out (B, T, 2W), [final states, each (2L, B, width) in the same order]).

    The reverse direction of a layer sees its input reversed in time and returns its outputs reversed in time; the join
    kernel writes the next layer's input and, for its reverse direction, the same tensor reversed.  The reverse
    direction is issued on a side stream forked from the caller's current stream and joined back into it with events,
    so that the two directions of a layer run concurrently.  Autograd runs each backward on the stream of its forward,
    so the two directions' backward passes overlap as well, and it synchronises (and records) the gradients it hands
    from one stream to the other; the forward's own cross-stream tensors are recorded here.
    `dropout`: None, or (p, seed, offset): the joined (B, T, 2H) output of every layer but the last is masked (boundary =
    layer index) before the next layer's two directions read it; the reverse direction sees the masked values reversed
    in time.
    `lengths`: None, or per-row lengths (DESIGN.md §4.22), which `run` must pass on to its one-layer calls: every row is
    reversed over its own length, so the reverse direction starts at step len_b - 1; outputs are 0 past the length."""
    if x.dim() != 3:
        raise ValueError("input must be (batch, seq_len, input_size), got shape %s" % (tuple(x.shape),))
    _require_cuda_f32("input", x)
    B = x.shape[0]
    for k, s in enumerate(states):
        if s is not None:
            shape = (2 * num_layers, B, (output_size or hidden_size) if k == 0 else hidden_size)
            _require_cuda_f32("state", s)
            if tuple(s.shape) != shape:
                raise ValueError("bidirectional states must have shape %s (2 * num_layers, batch, width), got %s"
                                 % (shape, tuple(s.shape)))
    dev = x.device
    if lengths is not None:
        lengths = check_lengths(lengths, B, x.shape[1], dev)
    with torch.cuda.device(dev):
        main = torch.cuda.current_stream(dev)
        side = _side_stream(dev)
        inp_f, inp_r = _BidirInputFunction.apply(lengths, x)
        finals = []
        for l in range(num_layers):
            st_f = [None if s is None else s[2 * l] for s in states]
            st_r = [None if s is None else s[2 * l + 1] for s in states]
            side.wait_stream(main)                      # fork: the reverse input and states are ready
            for t in [inp_r] + st_r:
                if t is not None:
                    t.record_stream(side)
            with torch.cuda.stream(side):
                res_r = run(l, 1, inp_r, *st_r)
            res_f = run(l, 0, inp_f, *st_f)
            main.wait_stream(side)                      # join
            for t in res_r:
                t.record_stream(main)
            last = l == num_layers - 1
            if last:
                out = _BidirJoinFunction.apply(True, lengths, res_f[0], res_r[0])
            elif dropout is not None and lengths is not None:
                # the dropout kernel's own reversal spans all T steps: reverse over each row's length separately
                inp_f = layer_dropout(_BidirJoinFunction.apply(True, lengths, res_f[0], res_r[0]), dropout, l)
                inp_r = _ReverseFunction.apply(lengths, inp_f)
            elif dropout is not None:
                inp_f, inp_r = layer_dropout(_BidirJoinFunction.apply(True, None, res_f[0], res_r[0]), dropout, l, rev=True)
            else:
                inp_f, inp_r = _BidirJoinFunction.apply(False, lengths, res_f[0], res_r[0])
            finals.append((res_f[1:], res_r[1:]))
    fin = [torch.stack([f[k] for pair in finals for f in pair]) for k in range(len(finals[0][0]))]
    return out, fin


class _TTLinearFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, shape: _lib.TTShape, n_in: int, n_out: int, x, bias, *cores):
        lib = _lib.load()
        _require_cuda_f32("input", x)
        for i, p in enumerate(cores):
            _require_cuda_f32("core %d" % i, p)
        if bias is not None:
            _require_cuda_f32("bias", bias)
        if x.dim() != 2 or x.shape[1] != n_in:
            raise ValueError("input must be (rows, %d), got %s" % (n_in, tuple(x.shape)))
        x = _dense16(x)
        rows = x.shape[0]
        with torch.cuda.device(x.device):
            blob = torch.cat([p.detach().reshape(-1) for p in cores])
            b = None if bias is None else bias.detach().contiguous()
            y = torch.empty((rows, n_out), device=x.device, dtype=torch.float32)
            stream = torch.cuda.current_stream(x.device).cuda_stream
            _lib.check(lib.ttrnn_ttlinear_forward(C.byref(shape), rows, _ptr(x), _ptr(blob), _ptr(b), _ptr(y),
                                                  None, stream), "ttrnn_ttlinear_forward")
        if any(ctx.needs_input_grad[3:]):
            ctx.shape, ctx.core_shapes, ctx.has_bias = shape, [tuple(p.shape) for p in cores], bias is not None
            ctx.save_for_backward(x, blob)
        return y

    @staticmethod
    def backward(ctx, dy):
        lib = _lib.load()
        x, blob = ctx.saved_tensors
        rows = x.shape[0]
        dy = _dense16(dy)
        with torch.cuda.device(x.device):
            nbytes = lib.ttrnn_ttlinear_workspace_bytes(C.byref(ctx.shape), rows)
            if nbytes < 0:
                raise RuntimeError("ttrnn_ttlinear_workspace_bytes failed: " + _lib.last_error())
            scratch = torch.empty(_bytes_to_floats(nbytes), device=x.device, dtype=torch.float32)
            d_x = torch.empty_like(x) if ctx.needs_input_grad[3] else None
            d_blob = torch.empty_like(blob)
            d_bias = torch.empty(dy.shape[1], device=x.device, dtype=torch.float32) \
                if (ctx.has_bias and ctx.needs_input_grad[4]) else None
            stream = torch.cuda.current_stream(x.device).cuda_stream
            _lib.check(lib.ttrnn_ttlinear_backward(C.byref(ctx.shape), rows, _ptr(x), _ptr(blob), _ptr(dy), _ptr(d_x),
                                                   _ptr(d_blob), _ptr(d_bias), _ptr(scratch), stream),
                       "ttrnn_ttlinear_backward")
        d_cores, off = [], 0
        for i, shp in enumerate(ctx.core_shapes):
            n = 1
            for v in shp:
                n *= v
            d_cores.append(d_blob[off:off + n].view(shp) if ctx.needs_input_grad[5 + i] else None)
            off += n
        return (None, None, None, d_x, d_bias) + tuple(d_cores)


def ttlinear(shape: _lib.TTShape, n_in: int, n_out: int, x: torch.Tensor, bias: Optional[torch.Tensor],
             cores: Sequence[torch.Tensor]) -> torch.Tensor:
    return _TTLinearFunction.apply(shape, n_in, n_out, x, bias, *cores)


class _CellStepFunction(torch.autograd.Function):
    """Gate math + state update of ONE timestep from the two pre-activation blocks (cell-step mode:
    is_naive / log_grads).  Reference: lstm.py:26-32, gru.py:33-44; backward = SURVEY.md 8a-10."""

    @staticmethod
    def forward(ctx, cell: str, c_grad_hook, a, u, h_prev, c_prev):
        lib = _lib.load()
        for name, t in (("input projection", a), ("hidden projection", u), ("hx", h_prev)):
            _require_cuda_f32(name, t)
        lstm = cell == "lstm"
        if lstm:
            _require_cuda_f32("cx", c_prev)
        B, H = h_prev.shape
        G = 4 if lstm else 3
        if tuple(a.shape) != (B, G * H) or tuple(u.shape) != (B, G * H):
            raise ValueError("gate blocks must be (%d, %d), got %s and %s" % (B, G * H, tuple(a.shape), tuple(u.shape)))
        a, u, h_prev = a.contiguous(), u.contiguous(), h_prev.contiguous()
        c_prev = c_prev.contiguous() if lstm else None
        with torch.cuda.device(a.device):
            h = torch.empty_like(h_prev)
            c = torch.empty_like(h_prev) if lstm else None
            stream = torch.cuda.current_stream(a.device).cuda_stream
            _lib.check(lib.ttrnn_cell_forward(_lib.CELL_LSTM if lstm else _lib.CELL_GRU, B, H, _ptr(a), _ptr(u),
                                              _ptr(h_prev), _ptr(c_prev), _ptr(h), _ptr(c), stream),
                       "ttrnn_cell_forward")
        ctx.cell, ctx.c_grad_hook = cell, c_grad_hook
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(a, u, h_prev, c_prev)
        return (h, c) if lstm else h

    @staticmethod
    def backward(ctx, *grads):
        lib = _lib.load()
        a, u, h_prev, c_prev = ctx.saved_tensors
        lstm = ctx.cell == "lstm"
        dh = grads[0]
        dc = grads[1] if lstm else None
        B, H = h_prev.shape
        dh = None if dh is None else dh.contiguous()
        dc = None if dc is None else dc.contiguous()
        with torch.cuda.device(a.device):
            da, du = torch.empty_like(a), torch.empty_like(u)
            dh_prev = torch.empty_like(h_prev)
            dc_prev = torch.empty_like(h_prev) if lstm else None
            dc_total = torch.empty_like(h_prev) if (lstm and ctx.c_grad_hook is not None) else None
            stream = torch.cuda.current_stream(a.device).cuda_stream
            _lib.check(lib.ttrnn_cell_backward(_lib.CELL_LSTM if lstm else _lib.CELL_GRU, B, H, _ptr(a), _ptr(u),
                                               _ptr(h_prev), _ptr(c_prev), _ptr(dh), _ptr(dc), _ptr(da), _ptr(du),
                                               _ptr(dh_prev), _ptr(dc_prev), _ptr(dc_total), stream),
                       "ttrnn_cell_backward")
        if dc_total is not None:
            ctx.c_grad_hook(dc_total)      # total dL/dc_t, as a tensor hook on the reference's `cy` sees it
        return None, None, da, du, (None if lstm else dh_prev), dc_prev


def cell_step(cell: str, a: torch.Tensor, u: torch.Tensor, h_prev: torch.Tensor,
              c_prev: Optional[torch.Tensor] = None, c_grad_hook=None):
    """One LSTM / GRU step from a = W_ih x + b_ih and u = W_hh h + b_hh.  LSTM -> (h, c); GRU -> h.
    `c_grad_hook(grad)` (LSTM) is called during backward with the total gradient of c_t."""
    return _CellStepFunction.apply(cell, c_grad_hook, a, u, h_prev, c_prev)
