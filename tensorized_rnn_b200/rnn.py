"""TTLSTM / TTGRU: the nn.Module mirror of the reference's recurrent modules.

Constructor signatures, attribute names, sub-module names (`cell{i}.input_weights`,
`cell{i}.hidden_weights`), state_dict keys/shapes, `init_hidden`, `param_count` and the
forward contract (batch-first input, one shared initial state, outputs of the last layer +
final state of the last layer) follow reference tensorized_rnn/tt_lstm.py:6-62,
tensorized_rnn/lstm.py:44-135 and tensorized_rnn/gru.py:52-194.  The time loop, the TT
contractions and the gate math run in the CUDA library (one call per sequence).

Two execution modes, chosen per module:
  * fused (default): one C-ABI call per sequence -> persistent recurrent CUDA kernels;
  * cell-step: one cell call per (timestep, layer), as the reference's Python loop does
    (lstm.py:123-133), used when the reference feature needs per-step module calls:
    `is_naive=True` (one TT matrix per gate, tt_linearset.py:5-38; the gate blocks come from
    G batched TT-matvec kernel calls and a fused gate kernel, `ttrnn_cell_forward/backward`) and
    `log_grads=True` with `fused_logging = False` or outside a training forward (forward hooks on the
    cells + tensor hooks on h_t / c_t feeding `ActivGradLogger`, rnn_utils.py:42-215; each step is then
    one fused single-step call).
  A training forward of a `log_grads=True` module stays fused (`fused_logging`, the default): the sequence
  kernels keep every layer's h_t / c_t, the BPTT kernel writes the total gradient of h_t / c_t of every
  step, and one reduction per (layer, variable) turns them into the four logged statistics
  (`ttrnn_rnn_backward_logged`, `ttrnn_step_norms`) that are appended to the same loggers.
  `new_core='first'/'last'` (rnn_utils.py:29-34) only changes the TT shapes and runs in either mode.

`bidirectional=True` (no reference counterpart; the contract of torch.nn.LSTM(bidirectional=True)) adds a reverse cell
per layer, `cell{i}_reverse`, and runs every (layer, direction) as a one-layer sequence call, the two directions of a
layer on two streams (functional.bidirectional_stack, DESIGN.md §4.17).  It needs the fused mode.

`dropout=p` (no reference counterpart; the contract of torch.nn.LSTM(dropout=p)): in training mode the output sequence of
every layer but the last is multiplied by a Bernoulli(1 - p) mask / (1 - p) before the next layer reads it, inside the
stack call (DESIGN.md §4.18).  It needs the fused mode as well.

`proj_size=P` (TTLSTM only; the contract of torch.nn.LSTM(proj_size=P)): each cell gets `projection_weights`, a TTLinear
H -> P without bias created after `hidden_weights`, and outputs h_t = W_hr (o_t * tanh(c_t)), which is also the next
step's hh input.  The recurrent kernels contract W_hr inside every step (DESIGN.md §4.19).  It needs the fused mode.

`forward` / `forward_states` also take a torch.nn.utils.rnn.PackedSequence, with torch's contract: the output is a
PackedSequence with the input's batch_sizes, sorted_indices and unsorted_indices, and the final states are those after
each sequence's own last step, in the caller's batch order.  The batch runs as one padded call with per-row lengths
(functional.rnn_sequence(lengths=...), DESIGN.md §4.22).  It needs the fused mode.
"""
from __future__ import annotations

import numbers
import warnings
from typing import List, Optional

import torch
from torch import nn

from torch.nn.utils.rnn import PackedSequence

from .functional import RnnSpec, bidirectional_stack, dropout_draw, pack_like, rnn_sequence, shared_bidirectional_state, \
    unpack_sequence
from .functional import cell_step
from .layers import TTLinear, TTLinearSet
from .rnn_utils import ActivGradLogger
from .shapes import tt_shape


def check_dropout(dropout, num_layers: int) -> float:
    """torch.nn.LSTM's validation of `dropout`: a number in [0, 1], with a warning when there is no layer boundary."""
    if isinstance(dropout, bool) or not isinstance(dropout, numbers.Number) or not 0 <= dropout <= 1:
        raise ValueError("dropout should be a number in range [0, 1] representing the probability of an element being "
                         "zeroed, got %r" % (dropout,))
    if dropout > 0 and num_layers == 1:
        warnings.warn("dropout option adds dropout after all but last recurrent layer, so non-zero dropout expects "
                      "num_layers greater than 1, but got dropout=%s and num_layers=%d" % (dropout, num_layers))
    return float(dropout)


def check_proj_size(proj_size, hidden_size: int) -> int:
    """torch.nn.LSTM's validation of `proj_size`: an int in [0, hidden_size)."""
    if isinstance(proj_size, bool) or not isinstance(proj_size, numbers.Integral) or proj_size < 0:
        raise ValueError("proj_size should be a positive integer or zero to disable projections, got %r" % (proj_size,))
    if proj_size >= hidden_size:
        raise ValueError("proj_size has to be smaller than hidden_size, got proj_size=%d, hidden_size=%d"
                         % (proj_size, hidden_size))
    return int(proj_size)


def active_dropout(module: nn.Module, device: torch.device):
    """(p, seed, offset) of this call's inter-layer dropout, or None: dropout > 0, training mode (also under no_grad, as
    torch.nn.LSTM), more than one layer.  Draws the mask from the device's CUDA generator."""
    if module.dropout > 0 and module.training and module.num_layers > 1:
        if device.type != "cuda":
            return (module.dropout, 0, 0)          # the engine rejects the CPU tensors itself
        seed, offset = dropout_draw(device)
        return (module.dropout, seed, offset)
    return None


class _StepLogSink(object):
    """Feeds ActivGradLogger from the fused path: (2, T) statistics per (layer, variable) instead of T hook calls.
    Same per-logger order as the reference's hooks: activations in time order (rnn_utils.py:139-140), gradients
    pushed to the left in reverse time (rnn_utils.py:149-150), i.e. in time order once the backward has finished."""

    def __init__(self, loggers):
        self.loggers = loggers           # per layer: {"h": logger, "c": logger (LSTM)}

    def activations(self, layer, var, stats):
        lg = self.loggers[layer].get(var)
        if lg is not None:
            lg.act.extend(stats[0].unbind(0))
            lg.log_act.extend(stats[1].unbind(0))

    def gradients(self, layer, var, stats):
        lg = self.loggers[layer].get(var)
        if lg is not None:
            lg.grad.extendleft(reversed(stats[0].unbind(0)))
            lg.log_grad.extendleft(reversed(stats[1].unbind(0)))


def param_count(matrix: nn.Module) -> int:
    """Number of weights in a module (reference tensorized_rnn/rnn_utils.py:300-310)."""
    assert isinstance(matrix, torch.nn.Module)
    return int(sum(p.shape.numel() for p in matrix.parameters()))


class _TTCellBase(nn.Module):
    n_gate = 0
    cell_kind = ""

    def __init__(self, input_size, hidden_size, bias, device, n_cores, tt_rank, is_naive=False, new_core=None, proj_size=0):
        super().__init__()
        assert new_core in [None, 'first', 'last']
        self.input_size = input_size
        self.hidden_size = hidden_size
        self.proj_size = proj_size
        self.bias = bias
        self.device = device
        self.n_cores = n_cores
        self.tt_rank = tt_rank
        self.is_naive = is_naive
        self.new_core = new_core
        # creation order (ih before hh) fixes the RNG stream, as in reference lstm.py:14-15
        self.input_weights = self._create_input_hidden_weights()
        self.hidden_weights = self._create_hidden_hidden_weights()
        if proj_size:
            # W_hr (H -> P, no bias), created last so that proj_size = 0 consumes the RNG as before.  new_core concerns
            # the gate axis, which the projection does not have
            self.projection_weights = TTLinear(out_features=proj_size, shape=tt_shape(hidden_size, proj_size, n_cores, 1),
                                               bias=False, auto_shapes=False, d=n_cores, tt_rank=tt_rank).to(device)

    # bias of the per-gate TTLinears of the naive form: the reference gives the TT-LSTM gates none
    # (tt_lstm.py:20,33) and the TT-GRU gates `self.bias` (gru.py:152,165)
    naive_bias_follows_flag = False

    def _tt_linear(self, in_features):
        if self.is_naive:
            return TTLinearSet(in_features=in_features, out_features=self.hidden_size, n_gates=self.n_gate,
                               bias=(self.bias if self.naive_bias_follows_flag else False), auto_shapes=True,
                               d=self.n_cores, tt_rank=self.tt_rank).to(self.device)
        shape = tt_shape(in_features, self.hidden_size, self.n_cores, self.n_gate, new_core=self.new_core)
        return TTLinear(out_features=self.n_gate * self.hidden_size, shape=shape, bias=self.bias,
                        auto_shapes=False, d=self.n_cores, tt_rank=self.tt_rank).to(self.device)

    def _create_input_hidden_weights(self):
        return self._tt_linear(self.input_size)

    def _create_hidden_hidden_weights(self):
        return self._tt_linear(self.proj_size or self.hidden_size)

    def flat_parameters(self) -> List[torch.Tensor]:
        """Parameters in C-ABI blob order: ih cores, ih bias, hh cores, hh bias (naive form: gate by gate), hr cores."""
        out: List[torch.Tensor] = []
        for w in (self.input_weights, self.hidden_weights):
            for lin in (list(w.gates) if self.is_naive else [w]):
                out += list(lin.weight_t.tt_cores)
                if lin.bias is not None:
                    out.append(lin.bias)
        if self.proj_size:
            out += list(self.projection_weights.weight_t.tt_cores)
        return out

    def _single_step_spec(self) -> RnnSpec:
        if getattr(self, "_step_spec", None) is None:
            self._step_spec = RnnSpec(self.cell_kind, self.input_size, self.hidden_size,
                                      self.input_weights.bias is not None,
                                      [self.input_weights.tt_modes()], [self.hidden_weights.tt_modes()],
                                      proj_size=self.proj_size,
                                      hr_shapes=[self.projection_weights.tt_modes()] if self.proj_size else None)
        return self._step_spec


class TTLSTMCell(_TTCellBase):
    """One TT-LSTM cell (reference tt_lstm.py:6-40; step semantics lstm.py:23-41)."""
    n_gate = 4
    cell_kind = "lstm"

    def forward(self, input, hx, cx):
        """One step: (h (B, P or H), c (B, H))."""
        hooked = hasattr(self, '_h_backward_hook')
        if self.is_naive or hooked:
            # two projections + the fused gate kernel.  The c_t hook of log_grads (reference lstm.py:35-39)
            # must see dL/dc_t INCLUDING the path through h_t = o*tanh(c_t), which is internal to the gate
            # kernel, so the kernel's backward hands that total to the hook.
            hy, cy = cell_step("lstm", self.input_weights(input), self.hidden_weights(hx), hx, cx,
                               c_grad_hook=getattr(self, '_c_backward_hook', None))
            if hooked and hy.requires_grad:
                assert hasattr(self, '_c_backward_hook')
                assert cy.requires_grad
                hy.register_hook(self._h_backward_hook)
        else:
            out, hy, cy = rnn_sequence(self._single_step_spec(), input.unsqueeze(1), hx, cx, self.flat_parameters())
        return hy, cy


class TTGRUCell(_TTCellBase):
    """One TT-GRU cell (reference gru.py:139-172; step semantics gru.py:25-50)."""
    n_gate = 3
    cell_kind = "gru"
    naive_bias_follows_flag = True

    def forward(self, input, hx):
        if self.is_naive:
            hy = cell_step("gru", self.input_weights(input), self.hidden_weights(hx), hx)
        else:
            out, hy = rnn_sequence(self._single_step_spec(), input.unsqueeze(1), hx, None, self.flat_parameters())
        if hasattr(self, '_h_backward_hook') and hy.requires_grad:      # reference gru.py:47-48
            hy.register_hook(self._h_backward_hook)
        return hy


class _TTRNNBase(nn.Module):
    cell_cls = None
    cell_kind = ""

    def __init__(self, input_size, hidden_size, num_layers, device, n_cores, tt_rank, bias=True,
                 is_naive=False, log_grads=False, new_core=None, bidirectional=False, dropout=0.0, proj_size=0):
        assert new_core in [None, 'first', 'last']
        if proj_size != 0 and self.cell_kind != "lstm":
            raise ValueError("proj_size argument is only supported for LSTM, not GRU")
        proj_size = check_proj_size(proj_size, hidden_size)
        if proj_size > 0 and (is_naive or log_grads):
            raise NotImplementedError("proj_size > 0 runs on the sequence kernels only; is_naive=True and log_grads=True "
                                      "need the cell-step mode, which has no projected form")
        if bidirectional and (is_naive or log_grads):
            raise NotImplementedError("bidirectional=True runs on the sequence kernels only; is_naive=True and "
                                      "log_grads=True need the cell-step mode, which has no bidirectional form")
        dropout = check_dropout(dropout, num_layers)
        if dropout > 0 and (is_naive or log_grads):
            raise NotImplementedError("dropout > 0 runs on the sequence kernels only; is_naive=True and log_grads=True "
                                      "need the cell-step mode, which has no dropout form")
        super().__init__()
        self.n_cores = n_cores
        self.tt_rank = tt_rank
        self.is_naive = is_naive
        self.new_core = new_core
        self.input_size = input_size
        self.hidden_size = hidden_size
        self.num_layers = num_layers
        self.bias = bias
        self.device = device
        self.log_grads = log_grads
        self.bidirectional = bool(bidirectional)
        self.dropout = dropout
        self.proj_size = proj_size
        self._all_layers = []
        for i in range(self.num_layers):
            cell = self._create_first_layer_cell() if i == 0 else self._create_other_layer_cell()
            setattr(self, 'cell{}'.format(i), cell)
            self._all_layers.append(cell)
            if self.bidirectional:
                # the reverse direction's cell of layer i, created right after the forward one (RNG order)
                cell = self._make_cell(cell.input_size)
                setattr(self, 'cell{}_reverse'.format(i), cell)
                self._all_layers.append(cell)
        self._spec: Optional[RnnSpec] = None
        # log_grads: keep training forwards on the sequence kernels (see the module docstring); False = the reference's
        # per-step hooks in cell-step mode
        self.fused_logging = True
        self._step_loggers = []
        if log_grads:
            self._install_loggers()

    def _install_loggers(self):
        """Per-layer loggers + hooks (reference lstm.py:66-80, gru.py:76-85): forward hooks on the cell
        modules, tensor-level backward hooks handed to the cells."""
        for i, cell in enumerate(self._all_layers):
            h_logger = ActivGradLogger("hidden_{}".format(i))
            h_forward, h_backward = h_logger.create_hooks(0)
            cell.register_forward_hook(h_forward)
            cell._h_backward_hook = h_backward
            self._step_loggers.append({"h": h_logger})
            if self.cell_kind == "lstm":
                c_logger = ActivGradLogger("cell_{}".format(i))
                c_forward, c_backward = c_logger.create_hooks(1)
                cell.register_forward_hook(c_forward)
                cell._c_backward_hook = c_backward
                self._step_loggers[-1]["c"] = c_logger

    def _fused_step_log(self):
        """The sink of the fused logging path, or None when this call must run step by step."""
        if not (self.log_grads and self.fused_logging) or self.is_naive or not torch.is_grad_enabled():
            return None
        if not any(p.requires_grad for p in self.parameters()):
            return None
        return _StepLogSink(self._step_loggers)

    @property
    def cell_step_mode(self) -> bool:
        """True when every (timestep, layer) is a separate cell call (is_naive / log_grads)."""
        return bool(self.is_naive or self.log_grads)

    def _make_cell(self, in_size):
        extra = {"proj_size": self.proj_size} if self.proj_size else {}
        return self.cell_cls(in_size, self.hidden_size, self.bias, self.device, n_cores=self.n_cores,
                             tt_rank=self.tt_rank, is_naive=self.is_naive, new_core=self.new_core, **extra)

    @property
    def output_size(self) -> int:
        """Width of every layer's output and of h: proj_size when projected, else hidden_size."""
        return self.proj_size or self.hidden_size

    def _create_first_layer_cell(self):
        return self._make_cell(self.input_size)

    def _create_other_layer_cell(self):
        return self._make_cell(2 * self.output_size if self.bidirectional else self.output_size)

    def param_count(self):
        total = 0
        for cell in self._all_layers:
            for attr in ('input_weights', 'hidden_weights', 'projection_weights'):
                if hasattr(cell, attr):
                    total += param_count(getattr(cell, attr))
        return total

    def spec(self) -> RnnSpec:
        if self.bidirectional:
            raise NotImplementedError("a bidirectional stack runs one-layer calls per (layer, direction); their "
                                      "descriptors are cell{l}[_reverse]._single_step_spec()")
        if self._spec is None:
            self._spec = RnnSpec(self.cell_kind, self.input_size, self.hidden_size, bool(self.bias),
                                 [c.input_weights.tt_modes() for c in self._all_layers],
                                 [c.hidden_weights.tt_modes() for c in self._all_layers],
                                 proj_size=self.proj_size,
                                 hr_shapes=[c.projection_weights.tt_modes() for c in self._all_layers] if self.proj_size
                                 else None)
        return self._spec

    def flat_parameters(self) -> List[torch.Tensor]:
        """Every cell's parameters in C-ABI blob order, cells in creation order (bidirectional: cell0, cell0_reverse,
        cell1, ...)."""
        out: List[torch.Tensor] = []
        for cell in self._all_layers:
            out += cell.flat_parameters()
        return out

    def _unpack(self, input):
        """(padded input, host lengths or None) of a forward input, which may be a PackedSequence."""
        if not isinstance(input, PackedSequence):
            return input, None
        if self.cell_step_mode:
            raise NotImplementedError("a PackedSequence runs on the sequence kernels only; is_naive=True and log_grads=True "
                                      "need the cell-step mode, which has no variable-length form")
        return unpack_sequence(input)

    def _check_input(self, input):
        if input.dim() != 3:
            raise ValueError("input must be (batch_size, seq_len, input_size)")
        if input.size(1) == 0:
            # the reference falls off its time loop with unbound locals (lstm.py:135 / gru.py:136)
            raise NameError("zero-length sequence: the reference raises NameError here and so does this module")

    def _run_bidirectional(self, input, states, lengths=None):
        """Bidirectional stack (functional.bidirectional_stack): every (layer, direction) is a one-layer sequence call.
        `states`: per state variable (2L, B, H) or None."""
        def run(layer, direction, x, h0, c0=None):
            cell = self._all_layers[2 * layer + direction]
            return rnn_sequence(cell._single_step_spec(), x, h0, c0, cell.flat_parameters(), lengths=lengths)

        return bidirectional_stack(input, states, self.num_layers, self.hidden_size, run,
                                   dropout=active_dropout(self, input.device), output_size=self.output_size,
                                   lengths=lengths)

    def _shared_to_bidirectional(self, input, state, width=None):
        return shared_bidirectional_state(state, self.num_layers, input.size(0), width or self.hidden_size)

    def _layer_states_in(self, input, states):
        """Per-layer initial states of the cell-step loop: a list of num_layers (batch, hidden) tensors per state
        variable; None = zeros."""
        shape = (self.num_layers, input.size(0), self.hidden_size)
        out = []
        for s in states:
            if s is None:
                s = torch.zeros(shape, device=input.device)
            elif tuple(s.shape) != shape:
                raise ValueError("per-layer states must have shape %s, got %s" % (shape, tuple(s.shape)))
            out.append(list(s.unbind(0)))
        return out


class TTLSTM(_TTRNNBase):
    """Drop-in for reference tensorized_rnn.tt_lstm.TTLSTM (tt_lstm.py:43-62)."""
    cell_cls = TTLSTMCell
    cell_kind = "lstm"

    def __init__(self, input_size, hidden_size, num_layers, device, n_cores, tt_rank, bias=True, is_naive=False,
                 log_grads=False, new_core=None, bidirectional=False, dropout=0.0, proj_size=0):
        super().__init__(input_size, hidden_size, num_layers, device, n_cores, tt_rank, bias=bias, is_naive=is_naive,
                         log_grads=log_grads, new_core=new_core, bidirectional=bidirectional, dropout=dropout,
                         proj_size=proj_size)

    def init_hidden(self, batch_size):
        h = torch.zeros(batch_size, self.output_size).to(self.device)
        c = torch.zeros(batch_size, self.hidden_size).to(self.device)
        return h, c

    def forward(self, input, init_states=None):
        """input (batch, seq_len, input_size) -> outputs (batch, seq_len, hidden), (h_T, c_T) of the last layer.
        `init_states` = (h0, c0), each (batch, hidden), shared by every layer; None = zeros.
        proj_size = P > 0: outputs and h are P wide, c stays hidden wide.
        bidirectional: outputs (batch, seq_len, 2 * hidden); (h0, c0) seed every layer and both directions; h_T, c_T
        are (2, batch, hidden): the last layer's forward direction after the last step, then its reverse direction
        after the first step.
        A PackedSequence input gives a PackedSequence output (see the module docstring)."""
        padded, lengths = self._unpack(input)
        out, st = self._forward_padded(padded, init_states, lengths)
        return (out if lengths is None else pack_like(out, lengths, input)), st

    def _forward_padded(self, input, init_states, lengths):
        """forward() on a padded batch: lengths None, or one length per row (outputs zero past them, the final states
        after each row's last step)."""
        self._check_input(input)
        if self.bidirectional:
            h0, c0 = (None, None) if init_states is None else init_states
            out, (h, c) = self._run_bidirectional(input, [self._shared_to_bidirectional(input, h0, self.output_size),
                                                          self._shared_to_bidirectional(input, c0)], lengths)
            return out, (h[-2:], c[-2:])
        sink = None if lengths is not None else self._fused_step_log()
        if self.cell_step_mode and sink is None:
            return self._forward_cell_steps(input, init_states)
        h0, c0 = (None, None) if init_states is None else init_states
        out, h, c = rnn_sequence(self.spec(), input, h0, c0, self.flat_parameters(), step_log=sink,
                                 dropout=active_dropout(self, input.device), lengths=lengths)
        return out, (h, c)

    def forward_states(self, input, states=None):
        """Per-layer states, the contract of torch.nn.LSTM: `states` = (h, c), each (num_layers, batch, hidden), or None
        (zeros).  Returns (outputs (batch, seq_len, hidden), (h_n, c_n)) with every layer's final state, each
        (num_layers, batch, hidden): feeding them to the next call continues the sequence exactly where this one
        stopped (streaming inference, truncated BPTT).  proj_size = P > 0: h and the outputs are P wide (as torch).
        bidirectional: the states are (2 * num_layers, batch, hidden), direction d of layer l at 2l + d, in and out, as
        torch.nn.LSTM(bidirectional=True) takes them; outputs are (batch, seq_len, 2 * hidden).
        A PackedSequence input gives a PackedSequence output (see the module docstring)."""
        packed = input
        input, lengths = self._unpack(input)
        self._check_input(input)
        if self.bidirectional:
            out, (h, c) = self._run_bidirectional(input, [None, None] if states is None else list(states), lengths)
            return (out if lengths is None else pack_like(out, lengths, packed)), (h, c)
        sink = None if lengths is not None else self._fused_step_log()
        if self.cell_step_mode and sink is None:
            return self._forward_cell_steps(input, states, layer_states=True)
        h0, c0 = (None, None) if states is None else states
        out, h, c = rnn_sequence(self.spec(), input, h0, c0, self.flat_parameters(), step_log=sink, layer_states=True,
                                 dropout=active_dropout(self, input.device), lengths=lengths)
        return (out if lengths is None else pack_like(out, lengths, packed)), (h, c)

    def _forward_cell_steps(self, input, init_states, layer_states=False):
        """The reference's own loop (lstm.py:116-135): step-major, layer-minor, one shared initial state
        (`layer_states`: one per layer, and every layer's final state is returned).
        Outputs are stacked at the end instead of written in place, which spares autograd the
        reference's T CopySlices nodes; values are identical."""
        batch_size, seq_len, _ = input.size()
        if layer_states:
            internal_state = list(zip(*self._layer_states_in(input, init_states if init_states is not None else (None, None))))
        else:
            if init_states is None:
                h = torch.zeros(batch_size, self.hidden_size, device=input.device)
                c = torch.zeros(batch_size, self.hidden_size, device=input.device)
            else:
                h, c = init_states
            internal_state = [(h, c)] * self.num_layers
        outputs = []
        for step in range(seq_len):
            x = input[:, step, :]
            for i, cell in enumerate(self._all_layers):
                (h, c) = internal_state[i]
                x, new_c = cell(x, h, c)
                internal_state[i] = (x, new_c)
            outputs.append(x)
        if layer_states:
            return torch.stack(outputs, dim=1), tuple(torch.stack(s) for s in zip(*internal_state))
        return torch.stack(outputs, dim=1), (x, new_c)


class TTGRU(_TTRNNBase):
    """Drop-in for reference tensorized_rnn.gru.TTGRU (gru.py:175-194)."""
    cell_cls = TTGRUCell
    cell_kind = "gru"

    def init_hidden(self, batch_size):
        return torch.zeros(batch_size, self.hidden_size).to(self.device)

    def forward(self, input, init_states=None):
        """input (batch, seq_len, input_size) -> outputs (batch, seq_len, hidden), h_T of the last layer.
        bidirectional: as for TTLSTM (outputs (batch, seq_len, 2 * hidden), h_T (2, batch, hidden)).
        A PackedSequence input gives a PackedSequence output (see the module docstring)."""
        padded, lengths = self._unpack(input)
        out, h = self._forward_padded(padded, init_states, lengths)
        return (out if lengths is None else pack_like(out, lengths, input)), h

    def _forward_padded(self, input, init_states, lengths):
        """forward() on a padded batch with optional per-row lengths (see TTLSTM._forward_padded)."""
        self._check_input(input)
        if self.bidirectional:
            out, (h,) = self._run_bidirectional(input, [self._shared_to_bidirectional(input, init_states)], lengths)
            return out, h[-2:]
        sink = None if lengths is not None else self._fused_step_log()
        if self.cell_step_mode and sink is None:
            return self._forward_cell_steps(input, init_states)
        out, h = rnn_sequence(self.spec(), input, init_states, None, self.flat_parameters(), step_log=sink,
                              dropout=active_dropout(self, input.device), lengths=lengths)
        return out, h

    def forward_states(self, input, states=None):
        """Per-layer states, the contract of torch.nn.GRU: `states` (num_layers, batch, hidden) or None (zeros).
        Returns (outputs (batch, seq_len, hidden), h_n (num_layers, batch, hidden)) with every layer's final state.
        bidirectional: states (2 * num_layers, batch, hidden), outputs (batch, seq_len, 2 * hidden), as torch.nn.GRU.
        A PackedSequence input gives a PackedSequence output (see the module docstring)."""
        packed = input
        input, lengths = self._unpack(input)
        self._check_input(input)
        if self.bidirectional:
            out, (h,) = self._run_bidirectional(input, [states], lengths)
            return (out if lengths is None else pack_like(out, lengths, packed)), h
        sink = None if lengths is not None else self._fused_step_log()
        if self.cell_step_mode and sink is None:
            return self._forward_cell_steps(input, states, layer_states=True)
        out, h = rnn_sequence(self.spec(), input, states, None, self.flat_parameters(), step_log=sink, layer_states=True,
                              dropout=active_dropout(self, input.device), lengths=lengths)
        return (out if lengths is None else pack_like(out, lengths, packed)), h

    def _forward_cell_steps(self, input, init_states, layer_states=False):
        """The reference's own loop (gru.py:119-136); `layer_states` as for TTLSTM."""
        batch_size, seq_len, _ = input.size()
        if layer_states:
            internal_state, = self._layer_states_in(input, (init_states,))
        else:
            h = torch.zeros(batch_size, self.hidden_size, device=input.device) if init_states is None else init_states
            internal_state = [h] * self.num_layers
        outputs = []
        for step in range(seq_len):
            x = input[:, step, :]
            for i, cell in enumerate(self._all_layers):
                x = cell(x, internal_state[i])
                internal_state[i] = x
            outputs.append(x)
        if layer_states:
            return torch.stack(outputs, dim=1), torch.stack(internal_state)
        return torch.stack(outputs, dim=1), x
