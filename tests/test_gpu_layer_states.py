"""Per-layer initial and final states (`forward_states`, C ABI flag TTRNN_WS_LAYER_STATES).

A stack with per-layer states takes h0 / c0 of shape (L, B, H), returns every layer's (h_n, c_n), lets an upstream
gradient of each layer's final state enter that layer's BPTT, and gives each layer's own d_h0 / d_c0.  Three checks run
over the kernel routes of the engine (static kernels with and without contracted cores, row groups, time chunks, the
runtime-shape kernels, a rank-one layer 0, a GRU, rank padding, the backward overlap, T = 1):

1. broadcast equivalence: the shared (B, H) state expanded to (L, B, H) gives bit-identical outputs, last-layer final
   state and parameter gradients to `forward(input, (h0, c0))`; the per-layer d_h0 summed over layers matches the old
   summed d_h0;
2. distinct per-layer states against the FP64 oracle run one layer at a time (tests/layer_states_ref.py), with an
   upstream gradient on every layer's final state;
3. chunked equivalence: the sequence cut into 2 and 3 pieces with the states carried matches one call, and two
   autograd-linked calls give the gradients of one call.

Bars: 1e-5 forward, 1e-4 gradients (norm-wise relative) against the oracle; 1e-6 / 1e-5 between chunked and whole runs.
"""
import io
from contextlib import contextmanager, redirect_stdout

import pytest
import torch

import tensorized_rnn_b200 as tr
from tensorized_rnn_b200 import _lib
from helpers import FWD_TOL, GRAD_TOL, oracle, quiet, rel_err
from layer_states_ref import gru_layer_states, lstm_layer_states
from test_gpu_round2 import DEV, assert_grads
from test_gpu_static_paths import _sd_from_layers

pytestmark = pytest.mark.gpu
DEFAULTS = {"chunk_steps": 0, "static_kernels": 1, "row_groups": 1, "merge_cores": 1}


@contextmanager
def options(**kw):
    lib = _lib.load()
    for k, v in kw.items():
        assert lib.ttrnn_set_option(k.encode(), int(v)) == 0, k
    try:
        yield lib
    finally:
        for k in kw:
            lib.ttrnn_set_option(k.encode(), DEFAULTS[k])


CASES = [
    # name, cell, I, H, L, d, r, B, T, options, input gradient
    ("cfg3_merge_cores_0", "lstm", 40, 256, 3, 3, 8, 24, 8, {"merge_cores": 0}, True),
    ("cfg3_merge_cores_1", "lstm", 40, 256, 3, 3, 8, 24, 8, {"merge_cores": 1}, True),
    ("cfg3_merge_cores_2", "lstm", 40, 256, 3, 3, 8, 24, 8, {"merge_cores": 2}, True),
    ("cfg3_row_groups", "lstm", 40, 256, 2, 3, 8, 40, 7, {"row_groups": 24}, True),
    ("cfg3_chunks", "lstm", 40, 256, 2, 3, 8, 16, 10, {"chunk_steps": 4}, True),
    ("cfg3_runtime_shape", "lstm", 40, 256, 2, 3, 8, 12, 6, {"static_kernels": 0}, True),
    ("cfg1_rank_one_L2", "lstm", 1, 256, 2, 2, 4, 20, 9, {}, True),
    ("cfg1_rank_one_L2_no_input_grad", "lstm", 1, 256, 2, 2, 4, 20, 9, {}, False),
    ("cfg2_gru_L2", "gru", 1, 256, 2, 2, 4, 20, 9, {}, False),
    ("cfg3alt_rank_padded_d2r2", "lstm", 40, 256, 3, 2, 2, 16, 6, {}, True),
    ("cfg3_overlap_L3", "lstm", 40, 256, 3, 3, 8, 8, 6, {}, True),
    ("cfg3_T1", "lstm", 40, 256, 2, 3, 8, 12, 1, {}, True),
    ("gru_T1", "gru", 16, 256, 2, 2, 4, 12, 1, {}, True),
]
IDS = [c[0] for c in CASES]


def make_pair(cell, I, H, L, d, r, seed=123):
    """FP64 oracle layers and our module (FP32, on the GPU) with the same parameters."""
    layers = oracle.random_layers(cell, I, H, L, d, r, bias=True, seed=seed, requires_grad=True, scale=1.5,
                                  dtype=torch.float64)
    m = quiet(tr.TTLSTM if cell == "lstm" else tr.TTGRU, I, H, L, torch.device("cpu"), n_cores=d, tt_rank=r)
    m.load_state_dict({k: v.float() for k, v in _sd_from_layers(layers).items()})
    return layers, m.to(DEV)


def inputs(cell, I, H, L, B, T, seed=7):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, T, I, generator=g, dtype=torch.float64)
    st = [0.5 * torch.randn(L, B, H, generator=g, dtype=torch.float64) for _ in range(2 if cell == "lstm" else 1)]
    w = [torch.randn(B, T, H, generator=g, dtype=torch.float64)] + \
        [torch.randn(L, B, H, generator=g, dtype=torch.float64) for _ in st]
    return x, st, w


def run_states(m, cell, x, states, w, want_dx=True):
    """forward_states + loss sum(out * w_out) + sum(h_n * w_h) (+ sum(c_n * w_c)); returns values and gradients."""
    for p in m.parameters():
        p.grad = None
    x = x.detach().clone().float().to(DEV).requires_grad_(want_dx)
    st = [s.detach().clone().float().to(DEV).requires_grad_(True) for s in states] if states is not None else None
    if cell == "lstm":
        out, (h, c) = m.forward_states(x, None if st is None else tuple(st))
        fin = [h, c]
    else:
        out, h = m.forward_states(x, None if st is None else st[0])
        fin = [h]
    loss = (out * w[0].float().to(DEV)).sum()
    for f, wf in zip(fin, w[1:]):
        loss = loss + (f * wf.float().to(DEV)).sum()
    loss.backward()
    torch.cuda.synchronize()
    return dict(out=out.detach(), fin=[f.detach() for f in fin], dx=x.grad if want_dx else None,
                dst=[s.grad for s in st] if st is not None else [],
                dp=[p.grad.clone() for p in m.flat_parameters()])


def oracle_states(layers, cell, x, states, w):
    for p in oracle.flat_params(layers):
        p.grad = None
    x = x.detach().clone().requires_grad_(True)
    st = [s.detach().clone().requires_grad_(True) for s in states]
    if cell == "lstm":
        out, fin = lstm_layer_states(oracle.lstm_forward, layers, x, st)
    else:
        out, fin = gru_layer_states(oracle.gru_forward, layers, x, st[0])
    loss = (out * w[0]).sum()
    for f, wf in zip(fin, w[1:]):
        loss = loss + (f * wf).sum()
    loss.backward()
    return dict(out=out.detach(), fin=[f.detach() for f in fin], dx=x.grad, dst=[s.grad for s in st],
                dp=[p.grad.clone() for p in oracle.flat_params(layers)])


def assert_matches_oracle(got, ref, want_dx=True):
    assert rel_err(got["out"], ref["out"]) <= FWD_TOL, rel_err(got["out"], ref["out"])
    for a, b in zip(got["fin"], ref["fin"]):
        assert a.shape == b.shape and rel_err(a, b) <= FWD_TOL, rel_err(a, b)
        for l in range(b.shape[0]):                     # every layer's final state, not only on average
            assert rel_err(a[l], b[l]) <= FWD_TOL, (l, rel_err(a[l], b[l]))
    if want_dx:
        assert rel_err(got["dx"], ref["dx"]) <= GRAD_TOL, rel_err(got["dx"], ref["dx"])
    for a, b in zip(got["dst"], ref["dst"]):
        for l in range(b.shape[0]):
            assert rel_err(a[l], b[l]) <= GRAD_TOL, (l, rel_err(a[l], b[l]))
    assert_grads(got["dp"], ref["dp"])


# ---- 1. broadcast equivalence ------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_broadcast_states_are_bit_identical_to_the_shared_contract(case):
    name, cell, I, H, L, d, r, B, T, opts, want_dx = case
    _, m = make_pair(cell, I, H, L, d, r)
    g = torch.Generator().manual_seed(3)
    x = torch.rand(B, T, I, generator=g).to(DEV)
    s0 = [(0.5 * torch.randn(B, H, generator=g)).to(DEV) for _ in range(2 if cell == "lstm" else 1)]
    w_out, w_h, w_c = (torch.randn(B, T, H, generator=g).to(DEV), torch.randn(B, H, generator=g).to(DEV),
                       torch.randn(B, H, generator=g).to(DEV))

    def run(per_layer):
        for p in m.parameters():
            p.grad = None
        xs = x.clone().requires_grad_(want_dx)
        st = [s.clone().requires_grad_(True) for s in s0]
        if per_layer:
            ex = [s.unsqueeze(0).expand(L, B, H) for s in st]
            res = m.forward_states(xs, tuple(ex) if cell == "lstm" else ex[0])
        else:
            res = m(xs, tuple(st) if cell == "lstm" else st[0])
        out = res[0]
        fin = list(res[1]) if cell == "lstm" else [res[1]]
        if per_layer:
            assert all(f.shape == (L, B, H) for f in fin)
            fin = [f[L - 1] for f in fin]                # no upstream gradient on the inner layers' final states
        loss = (out * w_out).sum() + (fin[0] * w_h).sum() + ((fin[1] * w_c).sum() if cell == "lstm" else 0)
        loss.backward()
        torch.cuda.synchronize()
        return out.detach(), [f.detach() for f in fin], xs.grad, [s.grad for s in st], \
            [p.grad.clone() for p in m.flat_parameters()]

    with options(**opts):
        shared = run(False)
        layer = run(True)
    assert torch.equal(shared[0], layer[0])
    assert all(torch.equal(a, b) for a, b in zip(shared[1], layer[1]))
    assert all(torch.equal(a, b) for a, b in zip(shared[4], layer[4]))
    if want_dx:
        assert torch.equal(shared[2], layer[2])
    # the per-layer d_h0 / d_c0 summed over layers (autograd of the expand) against the engine's own sum
    for a, b in zip(layer[3], shared[3]):
        assert rel_err(a, b) <= 1e-6, rel_err(a, b)


# ---- 2. distinct per-layer states against the oracle -------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_distinct_layer_states_match_oracle(case):
    name, cell, I, H, L, d, r, B, T, opts, want_dx = case
    layers, m = make_pair(cell, I, H, L, d, r)
    x, st, w = inputs(cell, I, H, L, B, T)
    ref = oracle_states(layers, cell, x, st, w)
    with options(**opts):
        if name == "cfg3_overlap_L3":
            # the backward of the inner layers forks its weight-gradient work onto the second stream
            plan = _lib.describe_plan(m.spec().desc(B, T), training=True)
            sms = torch.cuda.get_device_properties(0).multi_processor_count
            assert plan[0]["bwd_overlap"] == 1 and plan[0]["chunk_steps"] == T, plan[0]
            assert all(p["ih_route"] == "dense" for p in plan[2:]), plan
            assert all(sms - -(-B // p["bwd_rows"]) >= 24 for p in plan[1:]), plan
        if name == "cfg3_row_groups":
            assert _lib.describe_plan(m.spec().desc(B, T), training=True)[0]["row_groups"] == 2
        got = run_states(m, cell, x, st, w, want_dx)
        if T == 1:                                     # and without states (zeros)
            zeros = [torch.zeros_like(s) for s in st]
            ref0 = oracle_states(layers, cell, x, zeros, w)
            ref0["dst"] = []
            got0 = run_states(m, cell, x, None, w, want_dx)
    assert_matches_oracle(got, ref, want_dx)
    if T == 1:
        assert_matches_oracle(got0, ref0, want_dx)


def test_zero_states_equal_no_states():
    """`states=None` means zeros, in the forward and in every layer's final state."""
    cell, I, H, L, d, r, B, T = "lstm", 40, 256, 3, 3, 8, 12, 5
    _, m = make_pair(cell, I, H, L, d, r)
    x = torch.rand(B, T, I, generator=torch.Generator().manual_seed(1)).to(DEV)
    with torch.no_grad():
        o1, (h1, c1) = m.forward_states(x)
        z = torch.zeros(L, B, H, device=DEV)
        o2, (h2, c2) = m.forward_states(x, (z, z))
    assert torch.equal(o1, o2) and torch.equal(h1, h2) and torch.equal(c1, c2)


def test_shape_errors():
    _, m = make_pair("lstm", 40, 256, 2, 3, 8)
    x = torch.rand(4, 3, 40, device=DEV)
    with pytest.raises(ValueError):
        m.forward_states(x, (torch.zeros(4, 256, device=DEV), torch.zeros(4, 256, device=DEV)))
    with pytest.raises(ValueError):                    # forward() keeps the reference's (B, H) contract
        m(x, (torch.zeros(2, 4, 256, device=DEV), torch.zeros(2, 4, 256, device=DEV)))


# ---- 3. chunked equivalence ----------------------------------------------------------------------------------------
def _cuts(T, pieces):
    b = [round(i * T / pieces) for i in range(pieces + 1)]
    return [(b[i], b[i + 1]) for i in range(pieces) if b[i + 1] > b[i]]


@pytest.mark.parametrize("case", [c for c in CASES if c[8] >= 3], ids=[c[0] for c in CASES if c[8] >= 3])
def test_chunked_run_matches_one_call(case):
    name, cell, I, H, L, d, r, B, T, opts, want_dx = case
    _, m = make_pair(cell, I, H, L, d, r)
    x, st, w = inputs(cell, I, H, L, B, T)
    x = x.float().to(DEV)
    st = [s.float().to(DEV) for s in st]
    pack = (lambda s: tuple(s)) if cell == "lstm" else (lambda s: s[0])
    unpack = (lambda f: list(f)) if cell == "lstm" else (lambda f: [f])
    with options(**opts):
        with torch.no_grad():
            out1, fin1 = m.forward_states(x, pack(st))
            fin1 = unpack(fin1)
            for pieces in (2, 3):
                cur, outs = st, []
                for a, b in _cuts(T, pieces):
                    o, f = m.forward_states(x[:, a:b], pack(cur))
                    outs.append(o)
                    cur = unpack(f)
                out = torch.cat(outs, dim=1)
                assert rel_err(out, out1) <= 1e-6, (pieces, rel_err(out, out1))
                for a_, b_ in zip(cur, fin1):
                    assert rel_err(a_, b_) <= 1e-6, (pieces, rel_err(a_, b_))
        # truncated BPTT without detaching: two calls linked through the carried states, one loss
        ref = run_states(m, cell, x, st, w, want_dx)
        for p in m.parameters():
            p.grad = None
        xs = x.clone().requires_grad_(want_dx)
        ss = [s.clone().requires_grad_(True) for s in st]
        (a, b), (_, c) = _cuts(T, 2)
        o_a, f_a = m.forward_states(xs[:, a:b], pack(ss))
        o_b, f_b = m.forward_states(xs[:, b:c], f_a)
        loss = (torch.cat([o_a, o_b], dim=1) * w[0].float().to(DEV)).sum()
        for f, wf in zip(unpack(f_b), w[1:]):
            loss = loss + (f * wf.float().to(DEV)).sum()
        loss.backward()
        torch.cuda.synchronize()
    assert_grads([p.grad for p in m.flat_parameters()], ref["dp"], tol=1e-5)
    if want_dx:
        assert rel_err(xs.grad, ref["dx"]) <= 1e-5
    for s, dref in zip(ss, ref["dst"]):
        assert rel_err(s.grad, dref) <= 1e-5


# ---- check 2 for the other execution modes -------------------------------------------------------------------------
@pytest.mark.parametrize("cell", ["lstm", "gru"])
def test_fused_log_grads_with_layer_states(cell):
    """log_grads runs fused (whole-batch plan + per-layer states); values match the oracle, and the logged statistics
    equal those of the cell-step mode on the same call."""
    I, H, L, d, r, B, T = (40, 256, 2, 3, 8, 12, 6) if cell == "lstm" else (16, 256, 2, 2, 4, 12, 6)
    layers = oracle.random_layers(cell, I, H, L, d, r, bias=True, seed=9, requires_grad=True, scale=1.5, dtype=torch.float64)
    x, st, w = inputs(cell, I, H, L, B, T)
    ref = oracle_states(layers, cell, x, st, w)
    logs = {}
    for fused in (True, False):
        tr.ActivGradLogger.reset()
        with redirect_stdout(io.StringIO()):
            m = (tr.TTLSTM if cell == "lstm" else tr.TTGRU)(I, H, L, torch.device("cpu"), n_cores=d, tt_rank=r,
                                                            log_grads=True)
        m.load_state_dict({k: v.float() for k, v in _sd_from_layers(layers).items()})
        m = m.to(DEV)
        m.fused_logging = fused
        with options(row_groups=4):                    # the whole-batch flag must win over a forced split
            got = run_states(m, cell, x, st, w)
        assert_matches_oracle(got, ref)
        tr.ActivGradLogger.end_minibatch()
        tr.ActivGradLogger.end_epoch()
        logs[fused] = tr.ActivGradLogger.get_logs()
    tr.ActivGradLogger.reset()
    assert sorted(logs[True]) == sorted(logs[False]) and logs[True]
    for k in logs[True]:
        assert rel_err(logs[True][k], logs[False][k]) <= 1e-4, k


@pytest.mark.parametrize("cell", ["lstm", "gru"])
def test_naive_cell_steps_with_layer_states(cell):
    I, H, L, d, r, B, T = 16, 64, 2, 2, 3, 6, 5
    with redirect_stdout(io.StringIO()):
        m = (tr.TTLSTM if cell == "lstm" else tr.TTGRU)(I, H, L, torch.device("cpu"), n_cores=d, tt_rank=r, is_naive=True)
    layers = oracle.layers_from_state_dict(m.state_dict(), L, dtype=torch.float64, requires_grad=True)
    m = m.to(DEV)
    x, st, w = inputs(cell, I, H, L, B, T)
    ref = oracle_states(layers, cell, x, st, w)
    got = run_states(m, cell, x, st, w)
    assert_matches_oracle(got, ref)


@pytest.mark.parametrize("cell", ["lstm", "gru"])
def test_dense_modules_with_layer_states(cell):
    """Dense LSTM / GRU against the dense oracle run layer by layer (each layer from its own initial state)."""
    import dense_oracle
    I, H, L, B, T = 128, 128, 2, 6, 5
    torch.manual_seed(0)
    m = (tr.LSTM if cell == "lstm" else tr.GRU)(I, H, L, torch.device("cpu"))
    layers = dense_oracle.layers_from_state_dict({k: v.double() for k, v in m.state_dict().items()}, L, requires_grad=True)
    m = m.to(DEV)
    x, st, w = inputs(cell, I, H, L, B, T)
    xr = x.clone().requires_grad_(True)
    sr = [s.clone().requires_grad_(True) for s in st]
    if cell == "lstm":
        inp, fin = lstm_layer_states(dense_oracle.lstm_forward, layers, xr, sr)
    else:
        inp, fin = gru_layer_states(dense_oracle.gru_forward, layers, xr, sr[0])
    loss = (inp * w[0]).sum() + sum((f * wf).sum() for f, wf in zip(fin, w[1:]))
    loss.backward()
    ref = dict(out=inp.detach(), fin=[f.detach() for f in fin], dx=xr.grad, dst=[s.grad for s in sr],
               dp=[p.grad.clone() for p in dense_oracle.flat_params(layers)])
    got = run_states(m, cell, x, st, w)
    assert_matches_oracle(got, ref)
