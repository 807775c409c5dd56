"""Bidirectional TT-LSTM / TT-GRU and dense LSTM / GRU stacks (`bidirectional=True`, DESIGN.md §4.17).

1. One layer is bit-identical to two unidirectional one-layer modules holding the same parameters, the reverse one run
   on x.flip(1) and flipped back: outputs, final states, every parameter gradient, d_x = dxf + dxr.flip(1) and the state
   gradients, over the kernel routes (static kernels with merge_cores 0 / 1 / 2, cfg1's rank-one layer 0 with and
   without d_x, cfg2's GRU, rank padding, the runtime-shape kernels, forced time chunks, T = 1, the dense modules).
2. Two and three layers against the FP64 oracles composed per direction (tests/bidir_ref.py), with distinct initial
   states per (layer, direction) and upstream gradients on the output and on every final state.  Bars: 1e-5 forward,
   1e-4 gradients (norm-wise relative).
3. forward()'s shared (B, H) state equals forward_states with that state broadcast to (2L, B, H).
4. Streams: repeated steps, a non-default caller stream and no_grad inference give bit-identical results.
5. Shape and state errors.
"""
import pytest
import torch

import tensorized_rnn_b200 as tr
from tensorized_rnn_b200 import _lib
from helpers import FWD_TOL, GRAD_TOL, oracle, quiet, rel_err
from bidir_ref import bidir_forward, bidir_layers, flat_pairs
from test_gpu_layer_states import options

import dense_oracle

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
CLS = {("tt", "lstm"): tr.TTLSTM, ("tt", "gru"): tr.TTGRU, ("dense", "lstm"): tr.LSTM, ("dense", "gru"): tr.GRU}


def make(kind, cell, I, H, L, d=0, r=0, bidirectional=True, seed=11):
    torch.manual_seed(seed)
    kw = dict(n_cores=d, tt_rank=r) if kind == "tt" else {}
    return quiet(CLS[(kind, cell)], I, H, L, torch.device("cpu"), bidirectional=bidirectional, **kw)


def data(cell, I, H, L, B, T, seed=7):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, T, I, generator=g)
    st = [0.5 * torch.randn(2 * L, B, H, generator=g) for _ in range(2 if cell == "lstm" else 1)]
    w = [torch.randn(B, T, 2 * H, generator=g)] + [torch.randn(2 * L, B, H, generator=g) for _ in st]
    return x, st, w


def pack(cell, st):
    return tuple(st) if cell == "lstm" else st[0]


def unpack(cell, fin):
    return list(fin) if cell == "lstm" else [fin]


def run_bidir(m, cell, x, st, w, want_dx=True, stream=None):
    """forward_states + loss sum(out * w_out) + sum over final states of sum(f * w_f); values and gradients."""
    for p in m.parameters():
        p.grad = None
    xs = x.detach().clone().to(DEV).requires_grad_(want_dx)
    ss = [s.detach().clone().to(DEV).requires_grad_(True) for s in st]
    ws = [v.to(DEV) for v in w]
    if stream is not None:
        stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream) if stream is not None else torch.cuda.stream(torch.cuda.current_stream()):
        out, fin = m.forward_states(xs, pack(cell, ss))
        fin = unpack(cell, fin)
        loss = (out * ws[0]).sum() + sum((f * wf).sum() for f, wf in zip(fin, ws[1:]))
        loss.backward()
    torch.cuda.synchronize()
    return dict(out=out.detach(), fin=[f.detach() for f in fin], dx=xs.grad if want_dx else None,
                dst=[s.grad for s in ss], dp=[p.grad.clone() for p in m.flat_parameters()])


def assert_same(a, b, want_dx=True):
    assert torch.equal(a["out"], b["out"])
    assert all(torch.equal(u, v) for u, v in zip(a["fin"], b["fin"]))
    assert all(torch.equal(u, v) for u, v in zip(a["dst"], b["dst"]))
    assert all(torch.equal(u, v) for u, v in zip(a["dp"], b["dp"]))
    if want_dx:
        assert torch.equal(a["dx"], b["dx"])


# ---- 1. one layer: bit-identical to two unidirectional modules -----------------------------------------------------
L1_CASES = [
    # name, kind, cell, I, H, d, r, B, T, options, input gradient
    ("cfg3_merge_cores_0", "tt", "lstm", 40, 256, 3, 8, 24, 8, {"merge_cores": 0}, True),
    ("cfg3_merge_cores_1", "tt", "lstm", 40, 256, 3, 8, 24, 8, {"merge_cores": 1}, True),
    ("cfg3_merge_cores_2", "tt", "lstm", 40, 256, 3, 8, 24, 8, {"merge_cores": 2}, True),
    ("cfg1_rank_one", "tt", "lstm", 1, 256, 2, 4, 20, 9, {}, True),
    ("cfg1_rank_one_no_input_grad", "tt", "lstm", 1, 256, 2, 4, 20, 9, {}, False),
    ("cfg2_gru", "tt", "gru", 1, 256, 2, 4, 20, 9, {}, False),
    ("rank_padded_d2r2", "tt", "lstm", 40, 256, 2, 2, 16, 6, {}, True),
    ("cfg3_runtime_shape", "tt", "lstm", 40, 256, 3, 8, 12, 6, {"static_kernels": 0}, True),
    ("cfg3_chunks", "tt", "lstm", 40, 256, 3, 8, 16, 10, {"chunk_steps": 4}, True),
    ("cfg3_T1", "tt", "lstm", 40, 256, 3, 8, 12, 1, {}, True),
    ("dense_lstm", "dense", "lstm", 128, 128, 0, 0, 12, 7, {}, True),
    ("dense_gru", "dense", "gru", 128, 128, 0, 0, 12, 7, {}, True),
]


@pytest.mark.parametrize("case", L1_CASES, ids=[c[0] for c in L1_CASES])
def test_one_layer_is_two_unidirectional_layers(case):
    name, kind, cell, I, H, d, r, B, T, opts, want_dx = case
    m = make(kind, cell, I, H, 1, d, r)
    uni = []
    for prefix in ("cell0.", "cell0_reverse."):
        u = make(kind, cell, I, H, 1, d, r, bidirectional=False)
        u.load_state_dict({"cell0." + k[len(prefix):]: v for k, v in m.state_dict().items() if k.startswith(prefix)})
        uni.append(u.to(DEV))
    m = m.to(DEV)
    x, st, w = data(cell, I, H, 1, B, T)
    with options(**opts):
        got = run_bidir(m, cell, x, st, w, want_dx)
        ref = dict(fin=[], dst=[], dp=[])
        outs, dxs = [], []
        for dr, u in enumerate(uni):
            for p in u.parameters():
                p.grad = None
            xs = (x.flip(1) if dr else x).to(DEV).requires_grad_(want_dx)
            ss = [s[dr].to(DEV).requires_grad_(True) for s in st]
            out, fin = u(xs, pack(cell, ss))
            fin = unpack(cell, fin)
            out_w = w[0][..., dr * H:(dr + 1) * H].to(DEV)
            loss = (out * (out_w.flip(1) if dr else out_w)).sum() + \
                sum((f * wf[dr].to(DEV)).sum() for f, wf in zip(fin, w[1:]))
            loss.backward()
            outs.append(out.detach().flip(1) if dr else out.detach())
            ref["fin"].append(fin)
            ref["dst"].append([s.grad for s in ss])
            ref["dp"] += [p.grad for p in u.flat_parameters()]
            dxs.append(xs.grad)
        torch.cuda.synchronize()
    assert torch.equal(got["out"], torch.cat(outs, dim=2))
    for k in range(len(st)):
        assert torch.equal(got["fin"][k], torch.stack([ref["fin"][0][k], ref["fin"][1][k]]).detach())
        assert torch.equal(got["dst"][k], torch.stack([ref["dst"][0][k], ref["dst"][1][k]]))
    assert all(torch.equal(a, b) for a, b in zip(got["dp"], ref["dp"]))
    if want_dx:
        assert torch.equal(got["dx"], dxs[0] + dxs[1].flip(1))


# ---- 2. two and three layers against the oracle composition --------------------------------------------------------
DEEP_CASES = [
    # name, kind, cell, I, H, L, d, r, B, T, input gradient
    ("ttlstm_cfg3_L2", "tt", "lstm", 40, 256, 2, 3, 8, 16, 6, True),
    ("ttlstm_cfg3_L3", "tt", "lstm", 40, 256, 3, 3, 8, 12, 5, True),
    ("ttlstm_cfg1_rank_one_L2", "tt", "lstm", 1, 256, 2, 2, 4, 12, 7, True),
    ("ttgru_L2", "tt", "gru", 16, 256, 2, 2, 4, 12, 6, True),
    ("ttgru_L3", "tt", "gru", 16, 256, 3, 2, 4, 8, 5, True),
    ("dense_lstm_L2", "dense", "lstm", 128, 128, 2, 0, 0, 8, 6, True),
    ("dense_gru_L3", "dense", "gru", 128, 128, 3, 0, 0, 8, 5, True),
]


def oracle_run(kind, cell, m, L, x, st, w):
    if kind == "tt":
        pairs = bidir_layers(oracle.layers_from_state_dict, m.state_dict(), L, dtype=torch.float64, requires_grad=True)
        fwd = oracle.lstm_forward if cell == "lstm" else oracle.gru_forward
        params = oracle.flat_params(flat_pairs(pairs))
    else:
        sd = {k: v.detach().double().cpu() for k, v in m.state_dict().items()}
        pairs = bidir_layers(dense_oracle.layers_from_state_dict, sd, L, requires_grad=True)
        fwd = dense_oracle.lstm_forward if cell == "lstm" else dense_oracle.gru_forward
        params = dense_oracle.flat_params(flat_pairs(pairs))
    xs = x.double().requires_grad_(True)
    ss = [s.double().requires_grad_(True) for s in st]
    out, fin = bidir_forward(fwd, cell, pairs, xs, ss)
    loss = (out * w[0].double()).sum() + sum((f * wf.double()).sum() for f, wf in zip(fin, w[1:]))
    loss.backward()
    return dict(out=out.detach(), fin=[f.detach() for f in fin], dx=xs.grad, dst=[s.grad for s in ss],
                dp=[p.grad for p in params])


@pytest.mark.parametrize("case", DEEP_CASES, ids=[c[0] for c in DEEP_CASES])
def test_stack_matches_oracle_composition(case):
    name, kind, cell, I, H, L, d, r, B, T, want_dx = case
    m = make(kind, cell, I, H, L, d, r)
    x, st, w = data(cell, I, H, L, B, T)
    ref = oracle_run(kind, cell, m, L, x, st, w)
    got = run_bidir(m.to(DEV), cell, x, st, w, want_dx)
    assert got["out"].shape == (B, T, 2 * H)
    assert rel_err(got["out"], ref["out"]) <= FWD_TOL, rel_err(got["out"], ref["out"])
    for a, b in zip(got["fin"], ref["fin"]):
        assert a.shape == (2 * L, B, H)
        for i in range(2 * L):                         # every (layer, direction)
            assert rel_err(a[i], b[i]) <= FWD_TOL, (i, rel_err(a[i], b[i]))
    for a, b in zip(got["dst"], ref["dst"]):
        for i in range(2 * L):
            assert rel_err(a[i], b[i]) <= GRAD_TOL, (i, rel_err(a[i], b[i]))
    if want_dx:
        assert rel_err(got["dx"], ref["dx"]) <= GRAD_TOL, rel_err(got["dx"], ref["dx"])
    assert len(got["dp"]) == len(ref["dp"])
    for i, (a, b) in enumerate(zip(got["dp"], ref["dp"])):
        assert rel_err(a, b) <= GRAD_TOL, (i, tuple(b.shape), rel_err(a, b))


def test_upper_layer_of_the_cfg3_shape_takes_the_dense_ih_route():
    """Layers >= 1 of a bidirectional cfg3-shape stack have 2H = 512 inputs: the ih projection of their one-layer call
    forms W_ih densely and runs on the tensor cores."""
    m = make("tt", "lstm", 40, 256, 3, 3, 8)
    for l in (1, 2):
        for c in (getattr(m, "cell%d" % l), getattr(m, "cell%d_reverse" % l)):
            plan = _lib.describe_plan(c._single_step_spec().desc(640, 160), training=True)
            assert plan[1]["ih_route"] == "dense", plan


# ---- 3. forward(): one shared state ---------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,cell", [("tt", "lstm"), ("tt", "gru"), ("dense", "lstm")])
def test_shared_state_forward_is_the_broadcast_per_layer_call(kind, cell):
    I, H, L, d, r, B, T = (40, 256, 2, 3, 8, 12, 5) if kind == "tt" else (128, 128, 2, 0, 0, 8, 5)
    if cell == "gru":
        I, d, r = 16, 2, 4
    m = make(kind, cell, I, H, L, d, r).to(DEV)
    g = torch.Generator().manual_seed(3)
    x = torch.rand(B, T, I, generator=g).to(DEV)
    s0 = [(0.5 * torch.randn(B, H, generator=g)).to(DEV) for _ in range(2 if cell == "lstm" else 1)]
    w_out = torch.randn(B, T, 2 * H, generator=g).to(DEV)
    w_fin = [torch.randn(2, B, H, generator=g).to(DEV) for _ in s0]

    def run(per_layer):
        for p in m.parameters():
            p.grad = None
        st = [s.clone().requires_grad_(True) for s in s0]
        if per_layer:
            out, fin = m.forward_states(x, pack(cell, [s.unsqueeze(0).expand(2 * L, B, H) for s in st]))
            fin = [f[-2:] for f in unpack(cell, fin)]
        else:
            out, fin = m(x, pack(cell, st))
            fin = unpack(cell, fin)
            assert all(f.shape == (2, B, H) for f in fin)
        loss = (out * w_out).sum() + sum((f * wf).sum() for f, wf in zip(fin, w_fin))
        loss.backward()
        torch.cuda.synchronize()
        return out.detach(), [f.detach() for f in fin], [s.grad for s in st], [p.grad.clone() for p in m.flat_parameters()]

    shared, layer = run(False), run(True)
    assert torch.equal(shared[0], layer[0])
    assert all(torch.equal(a, b) for a, b in zip(shared[1], layer[1]))
    assert all(torch.equal(a, b) for a, b in zip(shared[3], layer[3]))
    for a, b in zip(shared[2], layer[2]):
        assert rel_err(a, b) <= 1e-6, rel_err(a, b)
    # d_h0 of the shared state is the sum of the 2L per-(layer, direction) gradients
    st = [s.clone().requires_grad_(True) for s in s0]
    per = [s.unsqueeze(0).expand(2 * L, B, H).clone().detach().requires_grad_(True) for s in st]
    for p in m.parameters():
        p.grad = None
    out, fin = m.forward_states(x, pack(cell, per))
    loss = (out * w_out).sum() + sum((f[-2:] * wf).sum() for f, wf in zip(unpack(cell, fin), w_fin))
    loss.backward()
    for a, p in zip(shared[2], per):
        assert rel_err(a, p.grad.sum(0)) <= 1e-6, rel_err(a, p.grad.sum(0))


# ---- 4. streams ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,cell", [("tt", "lstm"), ("tt", "gru"), ("dense", "lstm")])
def test_streams_repeat_caller_stream_and_inference(kind, cell):
    I, H, L, d, r, B, T = (40, 256, 3, 3, 8, 24, 8) if kind == "tt" else (128, 128, 2, 0, 0, 8, 6)
    if cell == "gru":
        I, d, r = 16, 2, 4
    m = make(kind, cell, I, H, L, d, r).to(DEV)
    x, st, w = data(cell, I, H, L, B, T)
    a = run_bidir(m, cell, x, st, w)
    b = run_bidir(m, cell, x, st, w)
    assert_same(a, b)
    c = run_bidir(m, cell, x, st, w, stream=torch.cuda.Stream(DEV))
    assert_same(a, c)
    with torch.no_grad():
        out, fin = m.forward_states(x.to(DEV), pack(cell, [s.to(DEV) for s in st]))
    torch.cuda.synchronize()
    assert torch.equal(out, a["out"])
    assert all(torch.equal(f, g) for f, g in zip(unpack(cell, fin), a["fin"]))


# ---- 5. errors ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["tt", "dense"])
def test_shape_and_state_errors(kind):
    I, H, L = (40, 256, 2) if kind == "tt" else (128, 128, 2)
    m = make(kind, "lstm", I, H, L, 3, 8).to(DEV)
    x = torch.rand(4, 3, I, device=DEV)
    z = lambda *s: torch.zeros(*s, device=DEV)                              # noqa: E731
    with pytest.raises(ValueError):                 # per-layer states of a unidirectional stack: (L, B, H)
        m.forward_states(x, (z(L, 4, H), z(L, 4, H)))
    with pytest.raises(ValueError):                 # forward() takes one (B, H) state
        m(x, (z(2 * L, 4, H), z(2 * L, 4, H)))
    with pytest.raises((ValueError, RuntimeError)):  # wrong input width (the dense call finds it in the blob size)
        m(torch.rand(4, 3, I + 1, device=DEV))
    with pytest.raises(ValueError):
        m(torch.rand(3, I, device=DEV))
    with pytest.raises(TypeError):
        m(torch.rand(4, 3, I, device=DEV, dtype=torch.float64))
    out, (h, c) = m(x)                              # still usable after the errors
    assert out.shape == (4, 3, 2 * H) and h.shape == (2, 4, H) and c.shape == (2, 4, H)
