"""Projected dense LSTM (`proj_size`, DESIGN.md §4.20) without a GPU: construction, the name mapping onto
torch.nn.LSTM(proj_size=P), the proj_size = 0 bit-identity, validation, SpeakerEncoder(proj_size) and the C-ABI surface
(the ttrnn_dense_rnn_*_proj symbols, ttrnn_dense_rnn_param_count_proj values and refusals)."""
import ctypes as C
import io
import os
import re
from contextlib import redirect_stdout

import pytest
import torch
from torch import nn

import tensorized_rnn_b200 as tr
from tensorized_rnn_b200 import _lib
from helpers import ROOT
from dense_proj_ref import torch_lstm, torch_names

CPU = torch.device("cpu")


def _make(seed=5, I=40, H=256, L=3, **kw):
    torch.manual_seed(seed)
    return tr.LSTM(I, H, L, CPU, **kw)


def _desc(m, B=8, T=5):
    return _lib.DenseDesc(_lib.CELL_LSTM, m.num_layers, m.input_size, m.hidden_size, int(m.bias), T, B)


# ---- construction ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bidirectional", [False, True])
@pytest.mark.parametrize("bias", [True, False])
def test_dense_proj_construction_names_shapes_and_counts(bidirectional, bias):
    I, H, P, L = 40, 256, 128, 3
    m = _make(I=I, H=H, L=L, proj_size=P, bias=bias, bidirectional=bidirectional)
    D = 2 if bidirectional else 1
    assert m.proj_size == P and m.output_size == P
    sd = m.state_dict()
    for l in range(L):
        for sfx in ("", "_reverse")[:D]:
            cell = getattr(m, "cell%d%s" % (l, sfx))
            pre = "cell%d%s." % (l, sfx)
            want = [pre + "input_weights.weight", pre + "hidden_weights.weight"] + \
                ([pre + "hidden_weights.bias"] if bias else []) + [pre + "projection_weights.weight"]
            assert [k for k in sd if k.startswith(pre)] == want
            assert cell.input_weights.weight.shape == (4 * H, I if l == 0 else D * P)
            assert cell.input_weights.bias is None                              # the reference's dense LSTM quirk
            assert cell.hidden_weights.weight.shape == (4 * H, P)
            assert cell.projection_weights.weight.shape == (P, H) and cell.projection_weights.bias is None
            assert cell.flat_parameters()[-1] is cell.projection_weights.weight
    assert m.param_count() == sum(p.numel() for p in m.parameters()) == sum(p.numel() for p in m.flat_parameters())
    h, c = m.init_hidden(3)
    assert h.shape == (3, P) and c.shape == (3, H)


@pytest.mark.parametrize("bidirectional", [False, True])
def test_dense_proj_state_dict_maps_onto_torch(bidirectional):
    """Every key of the module maps to a torch.nn.LSTM(proj_size) parameter of the same shape; torch's only other keys are
    the ih biases, which the dense LSTM cell does not have."""
    m = _make(H=256, L=2, proj_size=128, bidirectional=bidirectional)
    t = torch_lstm(m)
    tsd = t.state_dict()
    mapped = []
    for l in range(m.num_layers):
        for sfx in ("", "_reverse") if bidirectional else ("",):
            cell = getattr(m, "cell%d%s" % (l, sfx))
            for name, p in zip(torch_names(m, l, sfx), cell.flat_parameters()):
                assert tsd[name].shape == p.shape and torch.equal(tsd[name], p.detach().double())
                mapped.append(name)
    assert sorted(set(tsd) - set(mapped)) == sorted(k for k in tsd if k.startswith("bias_ih"))
    assert all(float(tsd[k].abs().sum()) == 0 for k in tsd if k.startswith("bias_ih"))


def test_dense_proj_size_zero_is_bit_identical_to_the_old_module():
    """proj_size = 0: the parameters are the reference's construction order, nn.Linear by nn.Linear, and the RNG stream
    afterwards is the same."""
    I, H, L = 40, 256, 3
    m = _make(seed=9, I=I, H=H, L=L, proj_size=0)
    r_m = torch.rand(3)
    torch.manual_seed(9)
    ref = []
    for l in range(L):
        ref.append(nn.Linear(I if l == 0 else H, 4 * H, False))
        ref.append(nn.Linear(H, 4 * H, True))
    r_ref = torch.rand(3)
    sd = m.state_dict()
    want = [t for lin in ref for t in (lin.weight, lin.bias) if t is not None]
    assert len(sd) == len(want) and all(torch.equal(a, b) for a, b in zip(sd.values(), want))
    assert torch.equal(r_m, r_ref)
    d = _make(seed=9, I=I, H=H, L=L)
    assert list(d.state_dict()) == list(sd) and all(torch.equal(d.state_dict()[k], sd[k]) for k in sd)
    assert m.proj_size == 0 and m.output_size == H and not hasattr(m.cell0, "projection_weights")


def test_dense_proj_size_validation():
    for bad in (-1, 1.5, "8", True, None, 256, 257):
        with pytest.raises(ValueError):
            _make(H=256, proj_size=bad)
    with pytest.raises(ValueError, match="only supported for LSTM"):
        tr.GRU(40, 256, 2, CPU, proj_size=128)
    assert tr.GRU(40, 256, 1, CPU, proj_size=0).hidden_size == 256
    with pytest.raises(NotImplementedError):
        _make(proj_size=128, log_grads=True)
    # the module accepts any P torch accepts; the engine refuses P % 128 != 0 at call time
    assert _make(H=256, proj_size=100).output_size == 100


def test_dense_proj_module_rejects_cpu_tensors():
    m = _make(L=2, proj_size=128)
    with pytest.raises(RuntimeError):
        m(torch.rand(2, 3, 40))
    with pytest.raises(RuntimeError):
        m.forward_states(torch.rand(2, 3, 40))


def test_speaker_encoder_proj_size():
    enc = tr.SpeakerEncoder(40, 768, 3, 256, CPU, proj_size=256)
    assert enc.rnn.proj_size == 256 and isinstance(enc.rnn, tr.LSTM)
    assert enc.linear.in_features == 256 and enc.linear.out_features == 256
    with redirect_stdout(io.StringIO()):
        tt = tr.SpeakerEncoder(40, 768, 3, 256, CPU, compression="tt", proj_size=256)
    assert isinstance(tt.rnn, tr.TTLSTM) and tt.rnn.proj_size == 256 and tt.linear.in_features_total == 256
    for compression in (None, "tt"):
        with pytest.raises(ValueError, match="only supported for LSTM"):
            with redirect_stdout(io.StringIO()):
                tr.SpeakerEncoder(40, 256, 2, 64, CPU, compression=compression, use_gru=True, proj_size=128)
    # proj_size = 0 builds what the reference signature builds
    torch.manual_seed(3)
    a = tr.SpeakerEncoder(40, 256, 2, 64, CPU)
    torch.manual_seed(3)
    b = tr.SpeakerEncoder(40, 256, 2, 64, CPU, proj_size=0)
    sa, sb = a.state_dict(), b.state_dict()
    assert list(sa) == list(sb) and all(torch.equal(sa[k], sb[k]) for k in sa)


# ---- C ABI ----------------------------------------------------------------------------------------------------------
def test_dense_proj_symbols_and_param_count():
    header = open(os.path.join(ROOT, "include", "ttrnn_b200.h")).read()
    lib = _lib.load()
    # each takes the arguments of its counterpart plus int32_t proj_size
    for name, base in (("ttrnn_dense_rnn_forward_proj", "ttrnn_dense_rnn_forward_ex"),
                       ("ttrnn_dense_rnn_backward_proj", "ttrnn_dense_rnn_backward_ex"),
                       ("ttrnn_dense_rnn_workspace_bytes_proj", "ttrnn_dense_rnn_workspace_bytes"),
                       ("ttrnn_dense_rnn_param_count_proj", "ttrnn_dense_rnn_param_count")):
        assert re.search(r"\b%s\s*\(" % name, header), name
        assert _lib.SYMBOLS[name][1] == _lib.SYMBOLS[base][1] + [C.c_int32]
        assert getattr(lib, name) is not None
    assert lib.ttrnn_abi_version() == _lib.ABI_VERSION == 4
    for I, H, P, L, bias in ((40, 768, 256, 3, True), (128, 256, 128, 2, False), (40, 512, 384, 1, True)):
        m = _make(I=I, H=H, L=L, proj_size=P, bias=bias)
        d = _desc(m)
        assert lib.ttrnn_dense_rnn_param_count_proj(C.byref(d), P) == sum(p.numel() for p in m.flat_parameters())
        assert lib.ttrnn_dense_rnn_param_count_proj(C.byref(d), P) == m.param_count()
        sb, wb = C.c_int64(0), C.c_int64(0)
        assert lib.ttrnn_dense_rnn_workspace_bytes_proj(C.byref(d), C.byref(sb), C.byref(wb), P) == 0
        assert sb.value > 0 and wb.value > 0
    # a bidirectional layer is a one-layer call
    m = _make(I=40, H=256, L=2, proj_size=128, bidirectional=True)
    d = _lib.DenseDesc(_lib.CELL_LSTM, 1, 256, 256, 1, 5, 8)
    assert lib.ttrnn_dense_rnn_param_count_proj(C.byref(d), 128) == sum(p.numel() for p in m.cell1_reverse.flat_parameters())


def test_dense_param_count_proj_refusals():
    lib = _lib.load()
    m = _make(I=40, H=256, L=2, proj_size=128)
    d = _desc(m)
    assert lib.ttrnn_dense_rnn_param_count_proj(C.byref(d), 128) > 0
    for P, msg in ((0, b"proj_size >= 1"), (-128, b"proj_size >= 1"), (256, b"[1, hidden_size)"), (384, b"[1, hidden_size)"),
                   (100, b"multiple of 128"), (192, b"multiple of 128")):
        assert lib.ttrnn_dense_rnn_param_count_proj(C.byref(d), P) == -1, P
        assert msg in lib.ttrnn_last_error(), (P, lib.ttrnn_last_error())
    gd = _lib.DenseDesc.from_buffer_copy(d)
    gd.cell = _lib.CELL_GRU
    assert lib.ttrnn_dense_rnn_param_count_proj(C.byref(gd), 128) == -1
    assert b"LSTM" in lib.ttrnn_last_error()
    sb, wb = C.c_int64(0), C.c_int64(0)
    assert lib.ttrnn_dense_rnn_workspace_bytes_proj(C.byref(d), C.byref(sb), C.byref(wb), 0) != 0
    assert lib.ttrnn_dense_rnn_workspace_bytes_proj(C.byref(gd), C.byref(sb), C.byref(wb), 128) != 0
    # the compute calls refuse before touching a buffer or the device
    nul = [None] * 10
    assert lib.ttrnn_dense_rnn_forward_proj(C.byref(d), *nul, 0, 0) != 0
    assert lib.ttrnn_dense_rnn_forward_proj(C.byref(gd), *nul, 0, 128) != 0
    assert lib.ttrnn_dense_rnn_forward_proj(C.byref(d), *nul, 0, 100) != 0
    assert lib.ttrnn_dense_rnn_backward_proj(C.byref(d), *([None] * 15), 0, 0) != 0
    assert lib.ttrnn_dense_rnn_backward_proj(C.byref(d), *([None] * 15), 0, 256) != 0
    # the unprojected stack's sizes and counts are unchanged by the new calls
    u = _make(I=40, H=256, L=2)
    assert lib.ttrnn_dense_rnn_param_count(C.byref(_desc(u))) == u.param_count()
