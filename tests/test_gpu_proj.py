"""Projected TT-LSTM (`proj_size`, DESIGN.md §4.19) on the GPU against the FP64 reference (tests/proj_ref.py, which
tests/test_proj_cpu.py pins against torch.nn.LSTM(proj_size=P)).

1. Per-layer states, every state and output with an upstream gradient, over d2 r4 / d3 r8 chains, L = 1, 2, 3,
   P = H/2 and P not a multiple of 4, the rank-one layer 0 (I = 1), forced time chunks, no bias, no input gradient, no
   initial states, the backward overlap off and the runtime-shape switch, the GE2E LSTMP width (H 768, P 256).
2. The shared-state forward(), a sequence cut into 2 and 3 pieces against one call, bidirectional L = 2, dropout p = 0.3
   with the engine's own mask, no_grad inference bit-identical to the training forward.
3. The refusals of the C ABI.
Bars: 1e-5 forward, 1e-4 gradients (norm-wise relative) against the reference.
"""
import ctypes as C

import pytest
import torch

import tensorized_rnn_b200 as tr
from tensorized_rnn_b200 import _lib
from helpers import FWD_TOL, GRAD_TOL, quiet, rel_err
from bidir_ref import bidir_forward
from dropout_ref import dropout_layer_states
from layer_states_ref import lstm_layer_states
from proj_ref import flat_params, lstmp_forward, random_layers, state_dict
from test_gpu_dropout import draw_state, engine_masks, gen
from test_gpu_layer_states import options

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")

CASES = [
    # name, I, H, P, L, d, r, B, T, options, bias, input gradient, initial states
    ("d2r4_L1", 40, 64, 32, 1, 2, 4, 12, 7, {}, True, True, True),
    ("d2r4_L2_P_odd", 40, 64, 30, 2, 2, 4, 9, 6, {}, True, True, True),
    ("d3r8_L3", 40, 256, 128, 3, 3, 8, 10, 6, {}, True, True, True),
    ("d3r8_L3_P_odd", 40, 256, 90, 3, 3, 8, 7, 5, {}, True, True, True),
    ("d3r8_L2_chunks", 40, 256, 128, 2, 3, 8, 8, 9, {"chunk_steps": 4}, True, True, True),
    ("d3r8_L2_nobias", 40, 256, 128, 2, 3, 8, 8, 5, {}, False, True, True),
    ("d3r8_L2_no_dx_no_states", 40, 256, 128, 2, 3, 8, 8, 5, {}, True, False, False),
    ("d3r8_L3_overlap_off", 40, 256, 128, 3, 3, 8, 8, 5, {"bwd_overlap": 0}, True, True, True),
    ("d3r8_L2_runtime_shape", 40, 256, 128, 2, 3, 8, 8, 5, {"static_kernels": 0}, True, True, True),
    ("d2r4_rank_one_L2", 1, 128, 64, 2, 2, 4, 10, 8, {}, True, True, True),
    ("d2r4_rank_one_L2_no_dx", 1, 128, 64, 2, 2, 4, 10, 8, {}, True, False, True),
    ("ge2e_d3r8_L3", 40, 768, 256, 3, 3, 8, 16, 4, {}, True, True, True),
]
IDS = [c[0] for c in CASES]
DEFAULTS = {"bwd_overlap": 1}


def make_pair(I, H, P, L, d, r, bias=True, seed=123, bidirectional=False):
    """FP64 reference layers and the module (FP32, on the GPU) with the same parameters.  Bidirectional: the layers are
    in module order (cell0, cell0_reverse, cell1, ...)."""
    D = 2 if bidirectional else 1
    in_sizes = [I] + [D * P] * (L - 1)
    layers = [random_layers(I, H, P, 1, d, r, bias=bias, seed=seed + 7 * i, requires_grad=True, scale=1.5,
                            in_sizes=[in_sizes[i // D]])[0] for i in range(D * L)]
    m = quiet(tr.TTLSTM, I, H, L, torch.device("cpu"), n_cores=d, tt_rank=r, bias=bias, proj_size=P,
              bidirectional=bidirectional)
    names = ["cell%d%s" % (i // D, "_reverse" if i % D else "") for i in range(D * L)]
    m.load_state_dict({k: v.float() for k, v in state_dict(layers, names).items()})
    return layers, m.to(DEV)


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


def run_reference(layers, x, states, w, compose):
    flat = flat_params(layers)
    for p in flat:
        p.grad = None
    x = x.detach().clone().requires_grad_(True)
    st = [s.detach().clone().requires_grad_(True) for s in states] if states is not None else None
    out, fin = compose(x, st)
    loss = (out * w[0]).sum() + sum((f * wf).sum() for f, wf in zip(fin, w[1:]))
    loss.backward()
    return dict(out=out.detach(), fin=[f.detach() for f in fin], dx=x.grad, dst=[s.grad for s in st] if st else [],
                dp=[p.grad.clone() for p in flat])


def assert_close(got, ref, want_dx=True):
    assert got["out"].shape == ref["out"].shape
    assert rel_err(got["out"], ref["out"]) <= FWD_TOL, rel_err(got["out"], ref["out"])
    for a, b in zip(got["fin"], ref["fin"]):
        assert a.shape == b.shape
        for l in range(b.shape[0]):
            assert rel_err(a[l], b[l]) <= FWD_TOL, (l, rel_err(a[l], b[l]))
    if want_dx:
        assert rel_err(got["dx"], ref["dx"]) <= GRAD_TOL, rel_err(got["dx"], ref["dx"])
    for a, b in zip(got["dst"], ref["dst"]):
        for l in range(b.shape[0]):
            assert rel_err(a[l], b[l]) <= GRAD_TOL, (l, rel_err(a[l], b[l]))
    assert len(got["dp"]) == len(ref["dp"])
    for i, (a, b) in enumerate(zip(got["dp"], ref["dp"])):
        assert a.shape == b.shape and rel_err(a, b) <= GRAD_TOL, (i, tuple(b.shape), rel_err(a, b))


# ---- 1. per-layer states against the reference ------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_proj_matches_reference(case):
    name, I, H, P, L, d, r, B, T, opts, bias, want_dx, with_states = case
    layers, m = make_pair(I, H, P, L, d, r, bias=bias)
    x, st, w = inputs(I, H, P, L, B, T)
    st = st if with_states else None
    ref = run_reference(layers, x, st, w, lambda xx, ss: lstm_layer_states(lstmp_forward, layers, xx, ss))
    with options(**{k: v for k, v in opts.items() if k in ("chunk_steps", "static_kernels")}):
        lib = _lib.load()
        for k, v in opts.items():
            if k in DEFAULTS:
                lib.ttrnn_set_option(k.encode(), v)
        try:
            got = run_engine(m, x, st, w, want_dx)
        finally:
            for k in opts:
                if k in DEFAULTS:
                    lib.ttrnn_set_option(k.encode(), DEFAULTS[k])
    assert_close(got, ref, want_dx)


# ---- 2. the other contracts -----------------------------------------------------------------------------------------
def test_proj_shared_state_forward_and_cell():
    I, H, P, L, B, T = 40, 256, 96, 3, 6, 5
    layers, m = make_pair(I, H, P, L, 3, 8)
    g = torch.Generator().manual_seed(2)
    x = torch.rand(B, T, I, generator=g, dtype=torch.float64)
    s0 = [0.5 * torch.randn(B, n, generator=g, dtype=torch.float64) for n in (P, H)]
    xd = x.float().to(DEV)
    out, (h, c) = m(xd, tuple(s.float().to(DEV) for s in s0))
    ref_out, (rh, rc) = lstmp_forward(layers, x, tuple(s0))
    assert out.shape == (B, T, P) and h.shape == (B, P) and c.shape == (B, H)
    assert rel_err(out, ref_out) <= FWD_TOL and rel_err(h, rh) <= FWD_TOL and rel_err(c, rc) <= FWD_TOL
    # one cell step: (h (B, P), c (B, H)) through the sequence call with T = 1
    hy, cy = m.cell0(xd[:, 0], s0[0].float().to(DEV), s0[1].float().to(DEV))
    rh1, rc1 = lstmp_forward(layers[:1], x[:, :1], tuple(s0))[1]
    assert hy.shape == (B, P) and cy.shape == (B, H)
    assert rel_err(hy, rh1) <= FWD_TOL and rel_err(cy, rc1) <= FWD_TOL


@pytest.mark.parametrize("pieces", [2, 3])
def test_proj_chunked_sequence_matches_one_call(pieces):
    I, H, P, L, B, T = 40, 256, 128, 2, 8, 9
    _, m = make_pair(I, H, P, L, 3, 8)
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


def test_proj_bidirectional_L2():
    I, H, P, L, B, T = 40, 256, 64, 2, 6, 5
    layers, m = make_pair(I, H, P, L, 3, 8, bidirectional=True)
    x, st, w = inputs(I, H, P, L, B, T, D=2)
    pairs = [(layers[2 * l], layers[2 * l + 1]) for l in range(L)]
    ref = run_reference(layers, x, st, w, lambda xx, ss: bidir_forward(lstmp_forward, "lstm", pairs, xx, ss))
    got = run_engine(m, x, st, w)
    assert got["out"].shape == (B, T, 2 * P) and got["fin"][0].shape == (2 * L, B, P)
    assert_close(got, ref)


def test_proj_dropout_matches_composition():
    I, H, P, L, B, T, p = 40, 256, 96, 3, 8, 6, 0.3
    layers, m = make_pair(I, H, P, L, 3, 8)
    m.dropout = p
    x, st, w = inputs(I, H, P, L, B, T)
    seed, offset = draw_state()
    got = run_engine(m, x, st, w)
    assert gen().get_offset() == offset + 4
    masks = engine_masks(p, seed, offset, L, B, T, P)
    ref = run_reference(layers, x, st, w, lambda xx, ss: dropout_layer_states(
        lstmp_forward, "lstm", layers, xx, [mk.double().cpu() for mk in masks], ss))
    assert_close(got, ref)


def test_proj_no_grad_inference_is_bit_identical():
    I, H, P, L, B, T = 40, 256, 128, 3, 8, 6
    _, m = make_pair(I, H, P, L, 3, 8)
    x, st, w = inputs(I, H, P, L, B, T)
    train = run_engine(m, x, st, w)
    with torch.no_grad():
        out, (h, c) = m.forward_states(x.float().to(DEV), tuple(s.float().to(DEV) for s in st))
    assert torch.equal(out, train["out"]) and torch.equal(h, train["fin"][0]) and torch.equal(c, train["fin"][1])


# ---- 3. refusals of the C ABI ---------------------------------------------------------------------------------------
def test_proj_abi_refusals():
    lib = _lib.load()
    m = quiet(tr.TTLSTM, 40, 64, 2, torch.device("cpu"), n_cores=2, tt_rank=4, proj_size=16)
    spec = m.spec()
    d, pj = spec.desc(4, 3), spec.proj()
    ws = _lib.RnnWorkspace()
    assert lib.ttrnn_rnn_workspace_bytes_ex(C.byref(d), _lib.WS_PROJ, C.byref(ws)) != 0
    assert lib.ttrnn_rnn_workspace_bytes_proj(C.byref(d), None, 0, C.byref(ws)) != 0
    gd = _lib.RnnDesc.from_buffer_copy(d)
    gd.cell = _lib.CELL_GRU
    assert lib.ttrnn_rnn_workspace_bytes_proj(C.byref(gd), C.byref(pj), 0, C.byref(ws)) != 0
    bad = _lib.RnnProj.from_buffer_copy(pj)
    bad.hr[0].in_modes[0] += 1
    assert lib.ttrnn_rnn_workspace_bytes_proj(C.byref(d), C.byref(bad), 0, C.byref(ws)) != 0
    _lib.check(lib.ttrnn_rnn_workspace_bytes_proj(C.byref(d), C.byref(pj), _lib.WS_PROJ, C.byref(ws)), "ws")
    # a projected plan is refused by every other entry point, before any buffer is touched
    nul = [None] * 10
    assert lib.ttrnn_rnn_forward(C.byref(d), C.byref(ws), *nul) != 0
    assert b"TTRNN_WS_PROJ" in lib.ttrnn_last_error()
    assert lib.ttrnn_rnn_backward(C.byref(d), C.byref(ws), *([None] * 15)) != 0
    assert lib.ttrnn_rnn_forward_dropout(C.byref(d), C.byref(ws), *nul, None) != 0
    assert lib.ttrnn_rnn_backward_dropout(C.byref(d), C.byref(ws), *([None] * 15), None) != 0
    assert lib.ttrnn_rnn_backward_logged(C.byref(d), C.byref(ws), *([None] * 17)) != 0
    # the _proj entry points refuse a NULL pj, a GRU descriptor and a plan without the flag
    assert lib.ttrnn_rnn_forward_proj(C.byref(d), C.byref(ws), *nul, None, None) != 0
    assert b"pj" in lib.ttrnn_last_error()
    assert lib.ttrnn_rnn_backward_proj(C.byref(d), C.byref(ws), *([None] * 15), None, None) != 0
    assert lib.ttrnn_rnn_forward_proj(C.byref(gd), C.byref(ws), *nul, C.byref(pj), None) != 0
    assert b"LSTM" in lib.ttrnn_last_error()
    plain = quiet(tr.TTLSTM, 40, 64, 2, torch.device("cpu"), n_cores=2, tt_rank=4).spec().desc(4, 3)
    ws2 = _lib.RnnWorkspace()
    _lib.check(lib.ttrnn_rnn_workspace_bytes_ex(C.byref(plain), 0, C.byref(ws2)), "ws")
    assert lib.ttrnn_rnn_forward_proj(C.byref(plain), C.byref(ws2), *nul, C.byref(pj), None) != 0
    assert b"TTRNN_WS_PROJ" in lib.ttrnn_last_error()
    assert lib.ttrnn_rnn_backward_proj(C.byref(plain), C.byref(ws2), *([None] * 15), C.byref(pj), None) != 0
