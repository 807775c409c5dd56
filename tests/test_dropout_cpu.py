"""Inter-layer dropout without a GPU: the reference composition the GPU tests compare against (tests/dropout_ref.py)
pinned against torch.nn.LSTM / GRU(dropout=p) in FP64 with torch's own masks, the modules' construction (default,
validation, warning, unchanged parameters) and the C-ABI surface (ttrnn_rnn_forward_dropout, ttrnn_rnn_backward_dropout,
ttrnn_dropout_apply, TTRNN_WS_DROPOUT)."""
import io
import os
import re
import warnings
from contextlib import redirect_stdout

import pytest
import torch
import torch.nn.functional as F

import tensorized_rnn_b200 as tr
from tensorized_rnn_b200 import _lib
from helpers import ROOT
from bidir_ref import bidir_layers
from dropout_ref import dropout_bidir_forward, dropout_layer_states

import dense_oracle

MODULES = [("TTLSTM", dict(n_cores=3, tt_rank=4)), ("TTGRU", dict(n_cores=2, tt_rank=2)), ("LSTM", {}), ("GRU", {})]


def _make(name, seed=5, I=40, H=64, L=3, **extra):
    kw = dict(dict(MODULES)[name])
    kw.update(extra)
    torch.manual_seed(seed)
    with redirect_stdout(io.StringIO()):
        return getattr(tr, name)(I, H, L, torch.device("cpu"), **kw)


def _torch_rnn(cell, layer_params, I, H, L, p, bidirectional):
    """torch.nn.LSTM / GRU(dropout=p, batch_first=True) in FP64 holding the dense oracle's parameters; layer_params: per
    layer a tuple of one (or, bidirectional, two) parameter dicts.  The dense LSTM cell has no ih bias: zero in torch."""
    m = (torch.nn.LSTM if cell == "lstm" else torch.nn.GRU)(I, H, L, batch_first=True, dropout=p,
                                                            bidirectional=bidirectional).double()
    with torch.no_grad():
        for l, pair in enumerate(layer_params):
            for d, q in enumerate(pair):
                sfx = "_l%d%s" % (l, "_reverse" if d else "")
                getattr(m, "weight_ih" + sfx).copy_(q["w_ih"])
                getattr(m, "weight_hh" + sfx).copy_(q["w_hh"])
                getattr(m, "bias_ih" + sfx).copy_(q["b_ih"] if q["b_ih"] is not None else torch.zeros_like(q["b_hh"]))
                getattr(m, "bias_hh" + sfx).copy_(q["b_hh"])
    return m


def _torch_masks(seed, p, L, B, T, F_):
    """The masks torch.nn.LSTM / GRU(dropout=p) draws in training mode under `seed`, recovered by running F.dropout on
    ones in the same order: one per layer boundary, on the layer output as torch keeps it internally, (T, B, F) in
    memory, viewed batch-first."""
    torch.manual_seed(seed)
    return [F.dropout(torch.ones(T, B, F_, dtype=torch.float64).transpose(0, 1), p, True) for _ in range(L - 1)]


@pytest.mark.parametrize("cell", ["lstm", "gru"])
@pytest.mark.parametrize("bidirectional", [False, True])
@pytest.mark.parametrize("p", [0.4, 1.0])
def test_reference_composition_matches_torch_dropout(cell, bidirectional, p):
    I, H, B, T, L = 5, 6, 3, 7, 3
    D = 2 if bidirectional else 1
    torch.manual_seed(0)
    mod = (tr.LSTM if cell == "lstm" else tr.GRU)(I, H, L, torch.device("cpu"), bidirectional=bidirectional)
    sd = {k: v.double() for k, v in mod.state_dict().items()}
    if bidirectional:
        layer_params = bidir_layers(dense_oracle.layers_from_state_dict, sd, L, requires_grad=True)
    else:
        layer_params = [(q,) for q in dense_oracle.layers_from_state_dict(sd, L, requires_grad=True)]
    ref = _torch_rnn(cell, layer_params, I, H, L, p, bidirectional)
    ref.train()
    g = torch.Generator().manual_seed(1)
    x = torch.rand(B, T, I, generator=g, dtype=torch.float64)
    st = [torch.randn(D * L, B, H, generator=g, dtype=torch.float64) for _ in range(2 if cell == "lstm" else 1)]
    w_out = torch.randn(B, T, D * H, generator=g, dtype=torch.float64)
    w_st = [torch.randn(D * L, B, H, generator=g, dtype=torch.float64) for _ in st]

    def loss_of(out, fin):
        return (out * w_out).sum() + sum((f * w).sum() for f, w in zip(fin, w_st))

    masks = _torch_masks(11, p, L, B, T, D * H)
    assert all(((m == 0) | (m == 1 / (1 - p) if p < 1 else m == 0)).all() for m in masks)
    forward = dense_oracle.lstm_forward if cell == "lstm" else dense_oracle.gru_forward
    xa, sa = x.clone().requires_grad_(True), [s.clone().requires_grad_(True) for s in st]
    if bidirectional:
        out_a, fin_a = dropout_bidir_forward(forward, cell, layer_params, xa, masks, sa)
    else:
        out_a, fin_a = dropout_layer_states(forward, cell, [q for (q,) in layer_params], xa, masks, sa)
    loss_of(out_a, fin_a).backward()
    xb, sb = x.clone().requires_grad_(True), [s.clone().requires_grad_(True) for s in st]
    torch.manual_seed(11)
    out_b, fin_b = ref(xb, tuple(sb) if cell == "lstm" else sb[0])
    fin_b = list(fin_b) if cell == "lstm" else [fin_b]
    loss_of(out_b, fin_b).backward()

    tol = dict(rtol=0, atol=1e-12)
    assert torch.isfinite(out_a).all() and torch.allclose(out_a, out_b, **tol)
    for a, b in zip(fin_a, fin_b):
        assert a.shape == (D * L, B, H) and torch.allclose(a, b, **tol)
    assert torch.allclose(xa.grad, xb.grad, **tol)
    for a, b in zip(sa, sb):
        assert torch.allclose(a.grad, b.grad, **tol)
    for l, pair in enumerate(layer_params):
        for d, q in enumerate(pair):
            sfx = "_l%d%s" % (l, "_reverse" if d else "")
            assert torch.allclose(q["w_ih"].grad, getattr(ref, "weight_ih" + sfx).grad, **tol)
            assert torch.allclose(q["w_hh"].grad, getattr(ref, "weight_hh" + sfx).grad, **tol)
            if p == 1.0 and l > 0:                       # the layers above the first see zero input
                assert torch.count_nonzero(q["w_ih"].grad) == 0
    # the masks matter: without them the composition differs from torch's training forward
    out_c, _ = (dropout_bidir_forward(forward, cell, layer_params, x, [torch.ones_like(m) for m in masks], st)
                if bidirectional else
                dropout_layer_states(forward, cell, [q for (q,) in layer_params], x, [torch.ones_like(m) for m in masks], st))
    assert not torch.allclose(out_c, out_b, **tol)


@pytest.mark.parametrize("name", [m[0] for m in MODULES])
def test_dropout_construction(name):
    m = _make(name)
    assert m.dropout == 0.0
    a = _make(name, dropout=0.3)
    assert a.dropout == 0.3
    # no RNG consumed, no parameter or key added: the same state_dict values under the same seed
    sa, sm = a.state_dict(), m.state_dict()
    assert list(sa) == list(sm) and all(torch.equal(sa[k], sm[k]) for k in sa)
    assert _make(name, dropout=1).dropout == 1.0 and _make(name, dropout=0).dropout == 0.0
    for bad in (-0.1, 1.5, float("nan"), True, "0.2", None):
        with pytest.raises(ValueError):
            _make(name, dropout=bad)
    with pytest.warns(UserWarning, match="num_layers greater than 1"):
        _make(name, L=1, dropout=0.2)
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        _make(name, L=1, dropout=0.0)
        _make(name, L=2, dropout=0.2)
    b = _make(name, dropout=0.25, bidirectional=True)
    assert b.dropout == 0.25 and b.bidirectional


@pytest.mark.parametrize("name", ["TTLSTM", "TTGRU"])
def test_dropout_needs_the_fused_mode(name):
    with pytest.raises(NotImplementedError):
        _make(name, is_naive=True, dropout=0.1)
    with pytest.raises(NotImplementedError):
        _make(name, log_grads=True, dropout=0.1)
    assert _make(name, is_naive=True, dropout=0.0).is_naive            # as before


@pytest.mark.parametrize("name", [m[0] for m in MODULES])
def test_dropout_module_rejects_cpu_tensors(name):
    m = _make(name, L=2, dropout=0.5)
    with pytest.raises(RuntimeError):
        m(torch.rand(2, 3, 40))
    m.eval()
    with pytest.raises(RuntimeError):
        m(torch.rand(2, 3, 40))


def test_dropout_symbols_are_exported_and_declared():
    header = open(os.path.join(ROOT, "include", "ttrnn_b200.h")).read()
    lib = _lib.load()
    for name, nargs in (("ttrnn_rnn_forward_dropout", 13), ("ttrnn_rnn_backward_dropout", 18), ("ttrnn_dropout_apply", 11)):
        assert re.search(r"\bint %s\s*\(" % name, header), name
        assert len(_lib.SYMBOLS[name][1]) == nargs
        assert getattr(lib, name) is not None
    assert re.search(r"#define TTRNN_WS_DROPOUT\s+%d\b" % _lib.WS_DROPOUT, header)
    assert "typedef struct ttrnn_dropout" in header
    assert _lib.Dropout.seed.offset == 8 and _lib.Dropout.offset.offset == 16 and __import__("ctypes").sizeof(_lib.Dropout) == 24
    assert lib.ttrnn_abi_version() == _lib.ABI_VERSION == 4
