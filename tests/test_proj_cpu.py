"""Projected TT-LSTM (`proj_size`) without a GPU: the reference the GPU tests compare against (tests/proj_ref.py) pinned
against torch.nn.LSTM(proj_size=P) in FP64, the modules' construction and validation, and the C-ABI surface
(TTRNN_WS_PROJ, ttrnn_rnn_proj, the _proj symbols, ttrnn_rnn_param_count_proj)."""
import ctypes as C
import io
import os
import re
from contextlib import redirect_stdout

import pytest
import torch

import tensorized_rnn_b200 as tr
from tensorized_rnn_b200 import _lib
from helpers import ROOT
from bidir_ref import bidir_forward
from layer_states_ref import lstm_layer_states
from proj_ref import flat_params, lstmp_forward, random_layers, torch_lstmp

TOL = dict(rtol=0, atol=1e-12)


def _make(seed=5, I=40, H=64, L=3, **extra):
    torch.manual_seed(seed)
    with redirect_stdout(io.StringIO()):
        return tr.TTLSTM(I, H, L, torch.device("cpu"), **dict(dict(n_cores=3, tt_rank=4), **extra))


# ---- the reference against torch ------------------------------------------------------------------------------------
CASES = [
    # L, bidirectional, per-layer states, H, P, bias
    (1, False, False, 12, 6, True),
    (3, False, True, 12, 6, True),
    (3, False, False, 12, 6, True),
    (2, False, True, 12, 5, False),          # P not a multiple of 4, no bias
    (2, True, True, 12, 6, True),
    (3, True, True, 8, 5, True),
]


@pytest.mark.parametrize("case", CASES, ids=["L%d_%s_%s_H%d_P%d_%s" % (c[0], "bi" if c[1] else "uni",
                                                                           "layer" if c[2] else "shared", c[3], c[4],
                                                                           "bias" if c[5] else "nobias") for c in CASES])
def test_reference_matches_torch_lstm_proj(case):
    L, bidir, layer_states, H, P, bias = case
    I, B, T, D = 5, 3, 6, 2 if case[1] else 1
    in_sizes = [I] + [D * P] * (L - 1)
    pairs = [tuple(random_layers(I, H, P, 1, 2, 3, bias=bias, seed=10 * l + d, requires_grad=True, scale=1.5,
                                 in_sizes=[in_sizes[l]])[0] for d in range(D)) for l in range(L)]
    flat = [t for pair in pairs for q in pair for t in flat_params([q])]
    g = torch.Generator().manual_seed(1)
    x = torch.rand(B, T, I, generator=g, dtype=torch.float64)
    if layer_states:
        st = [torch.randn(D * L, B, P, generator=g, dtype=torch.float64), torch.randn(D * L, B, H, generator=g, dtype=torch.float64)]
    else:
        st = [torch.randn(B, P, generator=g, dtype=torch.float64), torch.randn(B, H, generator=g, dtype=torch.float64)]
    w_out = torch.randn(B, T, D * P, generator=g, dtype=torch.float64)
    w_st = [torch.randn(D * L if layer_states else 1, B, n, generator=g, dtype=torch.float64) for n in (P, H)]

    def loss_of(out, fin):
        return (out * w_out).sum() + sum((f * w).sum() for f, w in zip(fin, w_st))

    def grads():
        gs = [p.grad.clone() for p in flat]
        for p in flat:
            p.grad = None
        return gs

    xa, sa = x.clone().requires_grad_(True), [s.clone().requires_grad_(True) for s in st]
    if bidir:
        out_a, fin_a = bidir_forward(lstmp_forward, "lstm", pairs, xa, sa)
    elif layer_states:
        out_a, fin_a = lstm_layer_states(lstmp_forward, [q for (q,) in pairs], xa, sa)
    else:
        out_a, (h, c) = lstmp_forward([q for (q,) in pairs], xa, tuple(sa))
        fin_a = [h.unsqueeze(0), c.unsqueeze(0)]
    loss_of(out_a, fin_a).backward()
    ga = grads()

    xb, sb = x.clone().requires_grad_(True), [s.clone().requires_grad_(True) for s in st]
    tst = sb if layer_states else [s.unsqueeze(0).expand(L, *s.shape) for s in sb]
    out_b, fin_b = torch_lstmp(pairs, xb, tst, I, H, P, bias=bias)
    fin_b = list(fin_b) if layer_states else [f[-1:] for f in fin_b]
    loss_of(out_b, fin_b).backward()
    gb = grads()

    assert out_a.shape == (B, T, D * P) and torch.allclose(out_a, out_b, **TOL)
    for a, b in zip(fin_a, fin_b):
        assert a.shape == b.shape and torch.allclose(a, b, **TOL)
    assert torch.allclose(xa.grad, xb.grad, **TOL)
    for a, b in zip(sa, sb):
        assert torch.allclose(a.grad, b.grad, **TOL)
    assert len(ga) == len(gb) == len(flat)
    for a, b in zip(ga, gb):
        assert torch.allclose(a, b, **TOL)
    assert all(float(t.abs().sum()) > 0 for t in ga)


# ---- construction ---------------------------------------------------------------------------------------------------
def test_proj_construction_names_shapes_and_counts():
    m = _make(H=64, L=3, proj_size=24)
    assert m.proj_size == 24 and m.output_size == 24
    sd = m.state_dict()
    for l in range(3):
        keys = [k for k in sd if k.startswith("cell%d." % l)]
        assert [k for k in keys if "projection" in k] == ["cell%d.projection_weights.parameters.%d" % (l, k) for k in range(3)]
        cell = getattr(m, "cell%d" % l)
        assert cell.projection_weights.bias is None
        assert cell.projection_weights.shape == tr.shapes.tt_shape(64, 24, 3, 1)
        assert cell.hidden_weights.shape[0] == tr.shapes.auto_shape(24, 3)     # W_hh: P -> 4H
        assert cell.input_size == (40 if l == 0 else 24)
        # blob order: ih cores, ih bias, hh cores, hh bias, hr cores
        flat = cell.flat_parameters()
        assert flat[-3:] == list(cell.projection_weights.weight_t.tt_cores)
    assert m.param_count() == sum(p.numel() for p in m.parameters()) == sum(p.numel() for p in m.flat_parameters())
    b = _make(H=64, L=2, proj_size=24, bidirectional=True)
    assert b.cell1.input_size == b.cell1_reverse.input_size == 48
    assert [k for k in b.state_dict() if "projection" in k and "reverse" in k][0] == \
        "cell0_reverse.projection_weights.parameters.0"
    assert b.init_hidden(3)[0].shape == (3, 24) and b.init_hidden(3)[1].shape == (3, 64)


def test_proj_size_zero_is_bit_identical_to_the_old_module():
    a, m = _make(seed=9), _make(seed=9, proj_size=0)
    sa, sm = a.state_dict(), m.state_dict()
    assert list(sa) == list(sm) and all(torch.equal(sa[k], sm[k]) for k in sa)
    assert m.proj_size == 0 and m.output_size == 64 and not hasattr(m.cell0, "projection_weights")
    assert m.spec().proj() is None
    # the RNG stream after construction is the same too
    _make(seed=9)
    r1 = torch.rand(3)
    _make(seed=9, proj_size=0)
    r2 = torch.rand(3)
    assert torch.equal(r1, r2)


def test_proj_size_validation():
    for bad in (-1, 1.5, "8", True, None, 64, 65):
        with pytest.raises(ValueError):
            _make(H=64, proj_size=bad)
    with pytest.raises(NotImplementedError):
        _make(proj_size=8, is_naive=True)
    with pytest.raises(NotImplementedError):
        _make(proj_size=8, log_grads=True)
    with pytest.raises(ValueError):
        with redirect_stdout(io.StringIO()):
            tr.TTGRU(40, 64, 2, torch.device("cpu"), n_cores=2, tt_rank=2, proj_size=8)
    assert _make(proj_size=63).proj_size == 63
    assert _make(is_naive=True, proj_size=0).is_naive                       # as before


def test_proj_module_rejects_cpu_tensors():
    m = _make(L=2, proj_size=16)
    with pytest.raises(RuntimeError):
        m(torch.rand(2, 3, 40))
    with pytest.raises(RuntimeError):
        m.forward_states(torch.rand(2, 3, 40))


# ---- C ABI ----------------------------------------------------------------------------------------------------------
def test_proj_symbols_struct_and_param_count():
    header = open(os.path.join(ROOT, "include", "ttrnn_b200.h")).read()
    lib = _lib.load()
    for name, nargs in (("ttrnn_rnn_forward_proj", 14), ("ttrnn_rnn_backward_proj", 19),
                        ("ttrnn_rnn_workspace_bytes_proj", 4), ("ttrnn_rnn_param_count_proj", 2)):
        assert re.search(r"\b%s\s*\(" % name, header), name
        assert len(_lib.SYMBOLS[name][1]) == nargs
        assert getattr(lib, name) is not None
    assert re.search(r"#define TTRNN_WS_PROJ\s+%d\b" % _lib.WS_PROJ, header)
    assert "typedef struct ttrnn_rnn_proj" in header
    assert _lib.RnnProj.hr.offset == 8 and C.sizeof(_lib.RnnProj) == 8 + _lib.MAX_LAYERS * C.sizeof(_lib.TTShape)
    assert lib.ttrnn_abi_version() == _lib.ABI_VERSION == 4
    for L, H, P, bidir in ((3, 768, 256, False), (2, 64, 30, False), (1, 64, 7, True)):
        m = _make(H=H, L=L, proj_size=P, bidirectional=bidir)
        cells = [m.cell0] if bidir else [m]
        for c in cells:
            spec = c._single_step_spec() if bidir else c.spec()
            d = spec.desc(8, 5)
            n = lib.ttrnn_rnn_param_count_proj(C.byref(d), C.byref(spec.proj()))
            assert n == sum(p.numel() for p in c.flat_parameters()), (n, _lib.last_error())
            # without the projection the descriptor is malformed (W_hh is 4H x P)
            assert lib.ttrnn_rnn_param_count(C.byref(d)) == -1


def test_param_count_proj_refusals():
    lib = _lib.load()
    m = _make(H=64, L=2, proj_size=16)
    spec = m.spec()
    d, pj = spec.desc(4, 3), spec.proj()
    assert lib.ttrnn_rnn_param_count_proj(C.byref(d), None) == -1
    bad = _lib.RnnProj.from_buffer_copy(pj)
    bad.hr[1].out_modes[0] += 1                                        # not P x H
    assert lib.ttrnn_rnn_param_count_proj(C.byref(d), C.byref(bad)) == -1
    assert b"hr TT matrix" in lib.ttrnn_last_error()
    bad = _lib.RnnProj.from_buffer_copy(pj)
    bad.proj_size = 64                                                 # P >= H
    assert lib.ttrnn_rnn_param_count_proj(C.byref(d), C.byref(bad)) == -1
    gd = _lib.RnnDesc.from_buffer_copy(d)
    gd.cell = _lib.CELL_GRU
    assert lib.ttrnn_rnn_param_count_proj(C.byref(gd), C.byref(pj)) == -1
    assert b"LSTM" in lib.ttrnn_last_error()
