"""Projected dense LSTM (`proj_size`, DESIGN.md §4.20) on the GPU against torch.nn.LSTM(proj_size=P, batch_first=True) on
the CPU in FP64, with the module's weights copied in through the state_dict mapping (tests/dense_proj_ref.py).

1. Per-layer states with an upstream gradient on every output and final state: L = 1, 2, 3; H 256 / P 128, H 512 / P 384
   and the GE2E width H 768 / P 256; B >= 128 (tensor-core per-step GEMMs) and B < 128 (FFMA); no bias; no initial
   states; input gradients where input_size % 128 == 0.
2. The shared-state forward() against forward_states(), a sequence cut into 2 and 3 pieces against one call, bidirectional
   L = 2, dropout p = 0.3 with the engine's own mask, no_grad inference bit-identical to the training forward, the
   engine's refusal of P % 128 != 0.
3. One SpeakerEncoder(compression=None, proj_size=256) training step against the same model built from torch modules.
Bars: 1e-5 forward, 1e-4 gradients (norm-wise relative).
"""
import os
import sys

import pytest
import torch
from torch import nn

import tensorized_rnn_b200 as tr
from tensorized_rnn_b200 import _lib
from helpers import FWD_TOL, GRAD_TOL, ROOT, rel_err
from dense_proj_ref import layer_forward, layers_params, torch_layers, torch_lstm, torch_params
from dropout_ref import dropout_layer_states
from test_gpu_dropout import draw_state, engine_masks, gen

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ge2e_oracle  # noqa: E402  (test infrastructure)

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
CPU = torch.device("cpu")

CASES = [
    # name, I, H, P, L, B, T, bias, initial states
    ("L1_H256_P128_B130", 128, 256, 128, 1, 130, 5, True, True),
    ("L2_H256_P128_B24", 128, 256, 128, 2, 24, 6, True, True),
    ("L3_H256_P128_B128", 128, 256, 128, 3, 128, 4, True, True),
    ("L3_H256_P128_I40_B20", 40, 256, 128, 3, 20, 5, True, True),
    ("L2_H512_P384_B16", 128, 512, 384, 2, 16, 4, True, True),
    ("L2_nobias_B136", 128, 256, 128, 2, 136, 4, False, True),
    ("L2_nobias_B16", 128, 256, 128, 2, 16, 5, False, True),
    ("L2_no_initial_states", 128, 256, 128, 2, 20, 5, True, False),
    ("ge2e_L3_H768_P256_B160", 40, 768, 256, 3, 160, 4, True, True),
    ("ge2e_L3_H768_P256_B12", 128, 768, 256, 3, 12, 5, True, True),
]


def make(I, H, P, L, bias=True, seed=11, bidirectional=False):
    torch.manual_seed(seed)
    return tr.LSTM(I, H, L, CPU, bias=bias, proj_size=P, bidirectional=bidirectional).to(DEV)


def inputs(I, H, P, L, B, T, D=1, seed=7):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, T, I, generator=g, dtype=torch.float64)
    st = [0.5 * torch.randn(D * L, B, n, generator=g, dtype=torch.float64) for n in (P, H)]
    w = [torch.randn(B, T, D * P, generator=g, dtype=torch.float64)] + \
        [torch.randn(D * L, B, n, generator=g, dtype=torch.float64) for n in (P, H)]
    return x, st, w


def run_engine(m, x, states, w, want_dx=True):
    for p in m.parameters():
        p.grad = None
    x = x.detach().clone().float().to(DEV).requires_grad_(want_dx)
    st = [s.detach().clone().float().to(DEV).requires_grad_(True) for s in states] if states is not None else None
    out, (h, c) = m.forward_states(x, None if st is None else tuple(st))
    loss = (out * w[0].float().to(DEV)).sum() + (h * w[1].float().to(DEV)).sum() + (c * w[2].float().to(DEV)).sum()
    loss.backward()
    torch.cuda.synchronize()
    return dict(out=out.detach(), fin=[h.detach(), c.detach()], dx=x.grad if want_dx else None,
                dst=[s.grad for s in st] if st is not None else [], dp=[p.grad.clone() for p in m.flat_parameters()])


def run_torch(x, states, w, compose, params):
    """compose(x, states) -> (out, [h_n, c_n]) on the CPU in FP64; params: its parameters in module order."""
    x = x.detach().clone().requires_grad_(True)
    st = [s.detach().clone().requires_grad_(True) for s in states] if states is not None else None
    out, fin = compose(x, st)
    loss = (out * w[0]).sum() + sum((f * wf).sum() for f, wf in zip(fin, w[1:]))
    loss.backward()
    return dict(out=out.detach(), fin=[f.detach() for f in fin], dx=x.grad, dst=[s.grad for s in st] if st else [],
                dp=[p.grad.clone() for p in params])


def whole_stack(t):
    def compose(x, st):
        out, (h, c) = t(x, None if st is None else tuple(st))
        return out, [h, c]
    return compose


def assert_close(got, ref, want_dx=True):
    assert got["out"].shape == ref["out"].shape
    assert rel_err(got["out"], ref["out"]) <= FWD_TOL, rel_err(got["out"], ref["out"])
    for a, b in zip(got["fin"], ref["fin"]):
        assert a.shape == b.shape
        for l in range(b.shape[0]):
            assert rel_err(a[l], b[l]) <= FWD_TOL, (l, rel_err(a[l], b[l]))
    if want_dx:
        assert rel_err(got["dx"], ref["dx"]) <= GRAD_TOL, rel_err(got["dx"], ref["dx"])
    assert len(got["dst"]) == len(ref["dst"])
    for a, b in zip(got["dst"], ref["dst"]):
        for l in range(b.shape[0]):
            assert rel_err(a[l], b[l]) <= GRAD_TOL, (l, rel_err(a[l], b[l]))
    assert len(got["dp"]) == len(ref["dp"])
    for i, (a, b) in enumerate(zip(got["dp"], ref["dp"])):
        assert a.shape == b.shape and rel_err(a, b) <= GRAD_TOL, (i, tuple(b.shape), rel_err(a, b))


# ---- 1. per-layer states against torch --------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_dense_proj_matches_torch(case):
    name, I, H, P, L, B, T, bias, with_states = case
    m = make(I, H, P, L, bias=bias)
    x, st, w = inputs(I, H, P, L, B, T)
    st = st if with_states else None
    want_dx = I % 128 == 0
    t = torch_lstm(m)
    ref = run_torch(x, st, w, whole_stack(t), torch_params(t, m))
    lib = _lib.load()
    lib.ttrnn_tc_launch_count(1)
    got = run_engine(m, x, st, w, want_dx)
    if B >= 128:
        assert int(lib.ttrnn_tc_launch_count(0)) > 0
    assert got["out"].shape == (B, T, P) and got["fin"][0].shape == (L, B, P) and got["fin"][1].shape == (L, B, H)
    assert_close(got, ref, want_dx)


# ---- 2. the other contracts -----------------------------------------------------------------------------------------
def test_dense_proj_shared_state_forward():
    """forward(): one (h0 (B, P), c0 (B, H)) seeds every layer, the last layer's final states come back; it is the
    per-layer call with the state repeated, bit for bit, and its state gradients are the sums over layers."""
    I, H, P, L, B, T = 128, 256, 128, 3, 12, 5
    m = make(I, H, P, L)
    g = torch.Generator().manual_seed(2)
    x = torch.rand(B, T, I, generator=g, dtype=torch.float64)
    s0 = [0.5 * torch.randn(B, n, generator=g, dtype=torch.float64) for n in (P, H)]
    w = [torch.randn(B, T, P, generator=g, dtype=torch.float64)] + [torch.randn(1, B, n, generator=g, dtype=torch.float64)
                                                                     for n in (P, H)]
    xd = x.float().to(DEV)
    sd = [s.float().to(DEV).requires_grad_(True) for s in s0]
    out, (h, c) = m(xd, tuple(sd))
    assert out.shape == (B, T, P) and h.shape == (B, P) and c.shape == (B, H)
    with torch.no_grad():
        o2, (h2, c2) = m.forward_states(xd, tuple(s.detach().unsqueeze(0).expand(L, *s.shape).contiguous() for s in sd))
    assert torch.equal(out, o2) and torch.equal(h, h2[-1]) and torch.equal(c, c2[-1])
    loss = (out * w[0].float().to(DEV)).sum() + (h * w[1][0].float().to(DEV)).sum() + (c * w[2][0].float().to(DEV)).sum()
    loss.backward()
    t = torch_lstm(m)

    def compose(xx, ss):
        out_t, (ht, ct) = t(xx, tuple(s.unsqueeze(0).expand(L, *s.shape) for s in ss))
        return out_t, [ht[-1:], ct[-1:]]
    ref = run_torch(x, s0, w, compose, torch_params(t, m))
    assert rel_err(out, ref["out"]) <= FWD_TOL and rel_err(h, ref["fin"][0]) <= FWD_TOL and rel_err(c, ref["fin"][1]) <= FWD_TOL
    for a, b in zip(sd, ref["dst"]):
        assert rel_err(a.grad, b) <= GRAD_TOL
    # no initial states: zeros
    out0, (h0, _) = m(xd)
    with torch.no_grad():
        rout, (rh, _) = t(x)
    assert rel_err(out0, rout) <= FWD_TOL and rel_err(h0, rh[-1]) <= FWD_TOL


@pytest.mark.parametrize("pieces", [2, 3])
def test_dense_proj_chunked_sequence_matches_one_call(pieces):
    I, H, P, L, B, T = 128, 256, 128, 2, 8, 9
    m = make(I, H, P, L)
    x, st, w = inputs(I, H, P, L, B, T)
    whole = run_engine(m, x, st, w)
    for p in m.parameters():
        p.grad = None
    xd = x.float().to(DEV).requires_grad_(True)
    s = tuple(t.float().to(DEV).requires_grad_(True) for t in st)
    cuts = [round(i * T / pieces) for i in range(pieces + 1)]
    outs, state = [], s
    for a, b in zip(cuts[:-1], cuts[1:]):
        o, state = m.forward_states(xd[:, a:b], state)
        outs.append(o)
    out = torch.cat(outs, dim=1)
    loss = (out * w[0].float().to(DEV)).sum() + (state[0] * w[1].float().to(DEV)).sum() + \
        (state[1] * w[2].float().to(DEV)).sum()
    loss.backward()
    assert rel_err(out, whole["out"]) <= 1e-6
    assert rel_err(state[0], whole["fin"][0]) <= 1e-6 and rel_err(state[1], whole["fin"][1]) <= 1e-6
    assert rel_err(xd.grad, whole["dx"]) <= 1e-5
    for a, b in zip(s, whole["dst"]):
        assert rel_err(a.grad, b) <= 1e-5
    for p, b in zip(m.flat_parameters(), whole["dp"]):
        assert rel_err(p.grad, b) <= 1e-5


def test_dense_proj_bidirectional_L2():
    I, H, P, L, B, T = 128, 256, 128, 2, 20, 5
    m = make(I, H, P, L, bidirectional=True)
    assert m.cell1.input_weights.weight.shape == (4 * H, 2 * P)
    x, st, w = inputs(I, H, P, L, B, T, D=2)
    t = torch_lstm(m)
    ref = run_torch(x, st, w, whole_stack(t), torch_params(t, m))
    got = run_engine(m, x, st, w)
    assert got["out"].shape == (B, T, 2 * P) and got["fin"][0].shape == (2 * L, B, P)
    assert_close(got, ref)
    # forward(): the shared (B, P) / (B, H) state seeds both directions of every layer
    out, (h, c) = m(x.float().to(DEV), (st[0][0].float().to(DEV), st[1][0].float().to(DEV)))
    assert out.shape == (B, T, 2 * P) and h.shape == (2, B, P) and c.shape == (2, B, H)


def test_dense_proj_dropout_matches_composition():
    I, H, P, L, B, T, p = 128, 256, 128, 3, 16, 6, 0.3
    m = make(I, H, P, L)
    m.dropout = p
    x, st, w = inputs(I, H, P, L, B, T)
    seed, offset = draw_state()
    got = run_engine(m, x, st, w)
    assert gen().get_offset() == offset + 4
    masks = engine_masks(p, seed, offset, L, B, T, P)
    layers = torch_layers(m)
    ref = run_torch(x, st, w, lambda xx, ss: dropout_layer_states(layer_forward, "lstm", layers, xx,
                                                                   [mk.double().cpu() for mk in masks], ss),
                    layers_params(layers, m))
    assert_close(got, ref)


def test_dense_proj_no_grad_inference_is_bit_identical():
    I, H, P, L, B, T = 128, 256, 128, 3, 130, 6
    m = make(I, H, P, L)
    x, st, w = inputs(I, H, P, L, B, T)
    train = run_engine(m, x, st, w)
    with torch.no_grad():
        out, (h, c) = m.forward_states(x.float().to(DEV), tuple(s.float().to(DEV) for s in st))
    assert torch.equal(out, train["out"]) and torch.equal(h, train["fin"][0]) and torch.equal(c, train["fin"][1])


def test_dense_proj_engine_refuses_unsupported_proj_size():
    m = make(40, 256, 100, 1)
    with pytest.raises(ValueError, match="multiple of 128"):
        m(torch.rand(4, 3, 40, device=DEV))


# ---- 3. the GE2E training step ---------------------------------------------------------------------------------------
def _torch_step(enc, x, S, U):
    """The model of `enc` built from torch modules, FP64 on the CPU: forward and backward of the GE2E loss.  Returns
    (embeddings, loss, parameters in the order enc.rnn.flat_parameters() + linear + similarity weight / bias)."""
    t = torch_lstm(enc.rnn)
    lin = nn.Linear(enc.linear.in_features, enc.linear.out_features).double()
    with torch.no_grad():
        lin.weight.copy_(enc.linear.weight)
        lin.bias.copy_(enc.linear.bias)
    sw, sb = (nn.Parameter(p.detach().double().clone()) for p in (enc.similarity_weight, enc.similarity_bias))
    _, (h_n, _) = t(x.double())
    emb = ge2e_oracle.embed_normalize(lin(h_n[-1]))
    loss = ge2e_oracle.loss(emb.view(S, U, -1), sw, sb)
    loss.backward()
    return emb.detach(), loss.detach(), torch_params(t, enc.rnn) + [lin.weight, lin.bias, sw, sb]


def test_speaker_encoder_dense_lstmp_training_step():
    """One training step of SpeakerEncoder(compression=None, proj_size=256): embeddings, loss, every gradient, the
    reference's do_gradient_ops (similarity gradients scaled, norm clipped) and one SGD step, against the same model built
    from torch modules in FP64.  Each speaker's utterances share a speaker-specific input pattern: with inputs that do not
    tell the speakers apart, every embedding is nearly the same at initialisation (loss ~ ln S) and the GE2E gradient is
    all cancellation, which even torch's own FP32 run cannot reproduce to 1e-4."""
    S, U, T, mel, H, L, E, P, lr = 4, 5, 12, 40, 512, 3, 64, 256, 0.01
    torch.manual_seed(21)
    enc = tr.SpeakerEncoder(mel, H, L, E, CPU, compression=None, proj_size=P)
    g = torch.Generator().manual_seed(4)
    x = (torch.randn(S, 1, 1, mel, generator=g) + 0.3 * torch.randn(S, U, T, mel, generator=g)).reshape(S * U, T, mel)
    emb_ref, loss_ref, ref_params = _torch_step(enc, x, S, U)

    enc = enc.to(DEV)
    emb = enc(x.to(DEV))
    loss, _ = enc.loss(emb.view(S, U, E))
    loss.backward()
    torch.cuda.synchronize()
    assert rel_err(emb, emb_ref) <= FWD_TOL
    assert abs(float(loss.detach()) - float(loss_ref)) <= FWD_TOL * abs(float(loss_ref))
    params = enc.rnn.flat_parameters() + [enc.linear.weight, enc.linear.bias, enc.similarity_weight, enc.similarity_bias]
    assert len(params) == len(ref_params) == len(list(enc.parameters()))
    bad = {}
    for i, (p, r) in enumerate(zip(params, ref_params)):
        if p is enc.similarity_bias:
            assert abs(float(p.grad)) < 1e-6            # exactly zero mathematically (softmax shift invariance)
            continue
        e = rel_err(p.grad, r.grad)
        if not e <= GRAD_TOL:
            bad[(i, tuple(p.shape))] = e
    assert not bad, bad

    # the reference's do_gradient_ops on both sides, then one SGD step
    enc.do_gradient_ops()
    ref_params[-2].grad *= 0.01
    ref_params[-1].grad *= 0.01
    torch.nn.utils.clip_grad_norm_(ref_params, enc.clip, norm_type=2)
    with torch.no_grad():
        for p, r in zip(params, ref_params):
            p -= lr * p.grad
            r -= lr * r.grad
    for p, r in zip(params, ref_params):
        assert rel_err(p, r) <= FWD_TOL
