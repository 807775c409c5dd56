"""Bidirectional stacks without a GPU: the reference composition the GPU tests compare against (tests/bidir_ref.py)
pinned against torch.nn.LSTM / GRU(bidirectional=True) in FP64, the modules' construction (cell names, shapes, input
sizes, RNG order, errors) and the C-ABI surface (ttrnn_time_reverse_add, ttrnn_bidir_join)."""
import io
import os
import re
from contextlib import redirect_stdout

import pytest
import torch

import tensorized_rnn_b200 as tr
from tensorized_rnn_b200 import _lib
from helpers import ROOT
from bidir_ref import bidir_forward, bidir_layers, flat_pairs

import dense_oracle


def _quiet(cls, *a, **k):
    with redirect_stdout(io.StringIO()):
        return cls(*a, **k)


def _torch_rnn(cell, pairs, I, H, L):
    """torch.nn.LSTM / GRU(bidirectional=True, batch_first=True) in FP64 holding the dense oracle's parameters.  The
    reference's dense LSTM cell has no ih bias, so torch's bias_ih is zero there."""
    m = (torch.nn.LSTM if cell == "lstm" else torch.nn.GRU)(I, H, L, batch_first=True, bidirectional=True).double()
    with torch.no_grad():
        for l, pair in enumerate(pairs):
            for d, p in enumerate(pair):
                sfx = "_l%d%s" % (l, "_reverse" if d else "")
                getattr(m, "weight_ih" + sfx).copy_(p["w_ih"])
                getattr(m, "weight_hh" + sfx).copy_(p["w_hh"])
                getattr(m, "bias_ih" + sfx).copy_(p["b_ih"] if p["b_ih"] is not None else torch.zeros_like(p["b_hh"]))
                getattr(m, "bias_hh" + sfx).copy_(p["b_hh"])
    return m


@pytest.mark.parametrize("cell", ["lstm", "gru"])
@pytest.mark.parametrize("L", [1, 3])
def test_reference_composition_matches_torch_bidirectional(cell, L):
    I, H, B, T = 5, 6, 3, 7
    torch.manual_seed(0)
    mod = (tr.LSTM if cell == "lstm" else tr.GRU)(I, H, L, torch.device("cpu"), bidirectional=True)
    sd = {k: v.double() for k, v in mod.state_dict().items()}
    pairs = bidir_layers(dense_oracle.layers_from_state_dict, sd, L, requires_grad=True)
    ref = _torch_rnn(cell, pairs, I, H, L)
    g = torch.Generator().manual_seed(1)
    x = torch.rand(B, T, I, generator=g, dtype=torch.float64)
    st = [torch.randn(2 * L, B, H, generator=g, dtype=torch.float64) for _ in range(2 if cell == "lstm" else 1)]
    w_out = torch.randn(B, T, 2 * H, generator=g, dtype=torch.float64)
    w_st = [torch.randn(2 * L, B, H, generator=g, dtype=torch.float64) for _ in st]

    def loss_of(out, fin):
        return (out * w_out).sum() + sum((f * w).sum() for f, w in zip(fin, w_st))

    xa, sa = x.clone().requires_grad_(True), [s.clone().requires_grad_(True) for s in st]
    out_a, fin_a = bidir_forward(dense_oracle.lstm_forward if cell == "lstm" else dense_oracle.gru_forward, cell, pairs,
                                 xa, sa)
    loss_of(out_a, fin_a).backward()
    xb, sb = x.clone().requires_grad_(True), [s.clone().requires_grad_(True) for s in st]
    out_b, fin_b = ref(xb, tuple(sb) if cell == "lstm" else sb[0])
    fin_b = list(fin_b) if cell == "lstm" else [fin_b]
    loss_of(out_b, fin_b).backward()

    tol = dict(rtol=0, atol=1e-12)
    assert out_a.shape == (B, T, 2 * H) and torch.allclose(out_a, out_b, **tol)
    for a, b in zip(fin_a, fin_b):
        assert a.shape == (2 * L, B, H) and torch.allclose(a, b, **tol)
    assert torch.allclose(xa.grad, xb.grad, **tol)
    for a, b in zip(sa, sb):
        assert torch.allclose(a.grad, b.grad, **tol)
    for l, pair in enumerate(pairs):
        for d, p in enumerate(pair):
            sfx = "_l%d%s" % (l, "_reverse" if d else "")
            assert torch.allclose(p["w_ih"].grad, getattr(ref, "weight_ih" + sfx).grad, **tol)
            assert torch.allclose(p["w_hh"].grad, getattr(ref, "weight_hh" + sfx).grad, **tol)
            assert torch.allclose(p["b_hh"].grad, getattr(ref, "bias_hh" + sfx).grad, **tol)
            if p["b_ih"] is not None:
                assert torch.allclose(p["b_ih"].grad, getattr(ref, "bias_ih" + sfx).grad, **tol)
    assert len(flat_pairs(pairs)) == 2 * L


TT_CASES = [("TTLSTM", dict(n_cores=3, tt_rank=4)), ("TTGRU", dict(n_cores=2, tt_rank=2)),
            ("LSTM", {}), ("GRU", {})]


def _make(name, bidirectional=None, seed=5, I=40, H=64, L=3, **extra):
    kw = dict(dict(TT_CASES)[name])
    kw.update(extra)
    if bidirectional is not None:
        kw["bidirectional"] = bidirectional
    torch.manual_seed(seed)
    return _quiet(getattr(tr, name), I, H, L, torch.device("cpu"), **kw)


@pytest.mark.parametrize("name", [c[0] for c in TT_CASES])
def test_bidirectional_cells_names_shapes_and_input_sizes(name):
    I, H, L = 40, 64, 3
    m = _make(name, True, I=I, H=H, L=L)
    uni = _make(name, False, I=I, H=H, L=L)
    names = [n for n, _ in m.named_children()]
    assert names == [n for l in range(L) for n in ("cell%d" % l, "cell%d_reverse" % l)]
    for l in range(L):
        for n in ("cell%d" % l, "cell%d_reverse" % l):
            c = getattr(m, n)
            assert c.input_size == (I if l == 0 else 2 * H) and c.hidden_size == H
        # the two directions of a layer have the same parameter shapes
        a = {k: v.shape for k, v in getattr(m, "cell%d" % l).state_dict().items()}
        b = {k: v.shape for k, v in getattr(m, "cell%d_reverse" % l).state_dict().items()}
        assert a == b
    sd = m.state_dict()
    assert set(sd) == set(uni.state_dict()) | {k.replace("cell%d." % l, "cell%d_reverse." % l)
                                               for k in uni.state_dict() for l in range(L) if k.startswith("cell%d." % l)}
    # layer 0 keeps the unidirectional shapes; layers >= 1 take 2H inputs
    for k, v in uni.state_dict().items():
        if k.startswith("cell0."):
            assert sd[k].shape == v.shape
    assert m.param_count() == sum(p.numel() for p in m.parameters())
    assert len(m.flat_parameters()) == len(list(m.parameters()))
    assert m.param_count() > 2 * _make(name, False, I=I, H=H, L=1).param_count()


@pytest.mark.parametrize("name", [c[0] for c in TT_CASES])
def test_bidirectional_false_is_the_unidirectional_module(name):
    """bidirectional=False builds what the constructor built before the flag existed: same keys, same values under a
    seed (same RNG consumption); with the flag set, cell0 is still the first thing created."""
    a = _make(name, None)
    b = _make(name, False)
    assert not b.bidirectional
    sa, sb = a.state_dict(), b.state_dict()
    assert list(sa) == list(sb) and all(torch.equal(sa[k], sb[k]) for k in sa)
    assert not any("reverse" in k for k in sa)
    c = _make(name, True)
    sc = c.state_dict()
    assert all(torch.equal(sa[k], sc[k]) for k in sa if k.startswith("cell0."))


@pytest.mark.parametrize("name", ["TTLSTM", "TTGRU"])
def test_bidirectional_constructor_errors_and_new_core(name):
    with pytest.raises(NotImplementedError):
        _make(name, True, is_naive=True)
    with pytest.raises(NotImplementedError):
        _make(name, True, log_grads=True)
    m = _make(name, True, new_core="first")                  # new_core only changes TT shapes
    assert m.cell1_reverse.input_size == 128
    with pytest.raises(NotImplementedError):                 # no whole-stack descriptor for a bidirectional stack
        m.spec()
    with pytest.raises(NotImplementedError):                 # dense baselines: as before
        _make(name.replace("TT", ""), True, log_grads=True)


def test_bidirectional_module_rejects_cpu_tensors():
    """No CPU fallback on the bidirectional path either."""
    for name in ("TTLSTM", "LSTM"):
        m = _make(name, True, L=2)
        with pytest.raises(RuntimeError):
            m(torch.rand(2, 3, 40))


def test_bidir_symbols_are_exported_and_declared():
    header = open(os.path.join(ROOT, "include", "ttrnn_b200.h")).read()
    lib = _lib.load()
    for name, nargs in (("ttrnn_time_reverse_add", 7), ("ttrnn_bidir_join", 9)):
        assert re.search(r"\bint %s\s*\(" % name, header), name
        assert len(_lib.SYMBOLS[name][1]) == nargs
        assert getattr(lib, name) is not None
    assert lib.ttrnn_abi_version() == _lib.ABI_VERSION == 4
