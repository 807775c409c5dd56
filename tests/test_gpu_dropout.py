"""Inter-layer dropout (`dropout=p`, DESIGN.md §4.18) on the GPU.

The mask the kernels used is read back from ttrnn_dropout_apply on a block of ones, with the (seed, offset) the module
draws from the CUDA generator, and fed to the FP64 oracle composition (tests/dropout_ref.py), which
tests/test_dropout_cpu.py pins against torch.nn.LSTM / GRU(dropout=p).

1. Every kernel route of tests/test_gpu_layer_states.py, plus a 444 + 196 row-group split of 640 rows (the mask is
   indexed by global row): outputs, every layer's final state, input, state and parameter gradients within 1e-5 / 1e-4.
2. Dropout off (p = 0, or any p in eval mode) is bit-identical to a module without the argument and draws nothing; the
   plan with TTRNN_WS_DROPOUT differs only by the masked buffers.
3. Mask properties: keep fraction, scalar and float4 paths agree, rows are global, successive calls differ, the seed
   reproduces a run, the generator offset advances by 4, no_grad in training mode masks as the training forward does.
4. p = 1: finite, zero ih core gradients above layer 0.
5. Bidirectional TT and dense stacks, dense LSTM / GRU against the reference composition.
"""
import ctypes as C

import pytest
import torch

import tensorized_rnn_b200 as tr
from tensorized_rnn_b200 import _lib
from helpers import FWD_TOL, GRAD_TOL, oracle, quiet, rel_err
from bidir_ref import bidir_layers, flat_pairs
from dropout_ref import dropout_bidir_forward, dropout_layer_states
from test_gpu_layer_states import CASES, assert_matches_oracle, inputs, make_pair, options, run_states

import dense_oracle

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
P = 0.25
SPLIT = ("cfg3_split_444_196", "lstm", 40, 256, 3, 3, 8, 640, 3, {"row_groups": 444}, True)
ALL_CASES = CASES + [SPLIT]


def gen():
    return torch.cuda.default_generators[0]


def draw_state():
    """(seed, offset) the next dropout call will draw."""
    return gen().initial_seed(), gen().get_offset()


def engine_masks(p, seed, offset, L, B, T, F):
    """mask / (1 - p) of boundaries 0 .. L-2 as the kernels apply it: ttrnn_dropout_apply on ones."""
    lib = _lib.load()
    dp = _lib.Dropout(p, 0, seed, offset)
    out = []
    for k in range(L - 1):
        ones = torch.ones(B, T, F, device=DEV)
        y = torch.empty_like(ones)
        _lib.check(lib.ttrnn_dropout_apply(B, T, F, 0, k, 0, C.byref(dp), ones.data_ptr(), y.data_ptr(), None,
                                           torch.cuda.current_stream().cuda_stream), "ttrnn_dropout_apply")
        out.append(y)
    torch.cuda.synchronize()
    return out


def oracle_dropout(layers, cell, x, st, w, masks):
    for p in oracle.flat_params(layers):
        p.grad = None
    x = x.detach().clone().requires_grad_(True)
    st = [s.detach().clone().requires_grad_(True) for s in st]
    fwd = oracle.lstm_forward if cell == "lstm" else oracle.gru_forward
    out, fin = dropout_layer_states(fwd, cell, layers, x, [m.double().cpu() for m in masks], st)
    loss = (out * w[0]).sum()
    for f, wf in zip(fin, w[1:]):
        loss = loss + (f * wf).sum()
    loss.backward()
    return dict(out=out.detach(), fin=[f.detach() for f in fin], dx=x.grad, dst=[s.grad for s in st],
                dp=[p.grad.clone() for p in oracle.flat_params(layers)])


# ---- 1. every route against the oracle composition ----------------------------------------------------------------
@pytest.mark.parametrize("case", ALL_CASES, ids=[c[0] for c in ALL_CASES])
def test_dropout_matches_oracle_composition(case):
    name, cell, I, H, L, d, r, B, T, opts, want_dx = case
    layers, m = make_pair(cell, I, H, L, d, r)
    m.dropout = P
    x, st, w = inputs(cell, I, H, L, B, T)
    with options(**opts):
        if name == SPLIT[0]:
            assert _lib.describe_plan(m.spec().desc(B, T), training=True)[0]["row_groups"] == 2
            lib = _lib.load()
            rows = (C.c_int64 * 2)()
            assert lib.ttrnn_rnn_row_groups(C.byref(m.spec().desc(B, T)), 0, rows) == 2 and tuple(rows) == (444, 196)
        seed, offset = draw_state()
        got = run_states(m, cell, x, st, w, want_dx)
        assert gen().get_offset() == offset + 4
    masks = engine_masks(P, seed, offset, L, B, T, H)
    kept = sum(float((mk != 0).float().mean()) for mk in masks) / len(masks)
    assert 0.5 < kept < 0.95, kept
    ref = oracle_dropout(layers, cell, x, st, w, masks)
    assert_matches_oracle(got, ref, want_dx)


# ---- 2. dropout off changes nothing -------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ALL_CASES, ids=[c[0] for c in ALL_CASES])
def test_dropout_off_is_bit_identical(case):
    name, cell, I, H, L, d, r, B, T, opts, want_dx = case
    _, m = make_pair(cell, I, H, L, d, r)
    x, st, w = inputs(cell, I, H, L, B, T)
    with options(**opts):
        base = run_states(m, cell, x, st, w, want_dx)
        runs = []
        for p, training in ((0.0, True), (P, False), (1.0, False)):
            m.dropout = p
            m.train(training)
            off = gen().get_offset()
            runs.append(run_states(m, cell, x, st, w, want_dx))
            assert gen().get_offset() == off                  # nothing drawn
        m.dropout = 0.0
        m.train()
    for got in runs:
        assert torch.equal(got["out"], base["out"])
        assert all(torch.equal(a, b) for a, b in zip(got["fin"], base["fin"]))
        assert all(torch.equal(a, b) for a, b in zip(got["dst"], base["dst"]))
        assert all(torch.equal(a, b) for a, b in zip(got["dp"], base["dp"]))
        if want_dx:
            assert torch.equal(got["dx"], base["dx"])


def test_plan_with_dropout_flag_only_adds_the_masked_buffers():
    lib = _lib.load()
    for L, B, T in ((3, 24, 8), (3, 640, 3), (1, 8, 4)):
        m = quiet(tr.TTLSTM, 40, 256, L, torch.device("cpu"), n_cores=3, tt_rank=8)
        desc = m.spec().desc(B, T)
        text = _lib.describe_plan(desc, training=True)
        a, b = _lib.RnnWorkspace(), _lib.RnnWorkspace()
        _lib.check(lib.ttrnn_rnn_workspace_bytes_ex(C.byref(desc), 0, C.byref(a)), "ws")
        _lib.check(lib.ttrnn_rnn_workspace_bytes_ex(C.byref(desc), _lib.WS_DROPOUT, C.byref(b)), "ws")
        assert _lib.describe_plan(desc, training=True) == text
        assert b.bwd_scratch_bytes == a.bwd_scratch_bytes
        groups = text[0].get("row_groups", 1)
        if L == 1:
            assert (b.saved_bytes, b.fwd_scratch_bytes) == (a.saved_bytes, a.fwd_scratch_bytes)
        elif groups == 1:
            assert b.saved_bytes - a.saved_bytes == (L - 1) * B * T * 256 * 4
            assert b.fwd_scratch_bytes - a.fwd_scratch_bytes == B * T * 256 * 4
        else:
            assert b.saved_bytes > a.saved_bytes and b.fwd_scratch_bytes > a.fwd_scratch_bytes
        assert sum(u != v for u, v in zip(a.plan, b.plan)) == 1           # the flag's own plan word
        # the plain entry points refuse a dropout plan; the dropout ones refuse p > 0 without it and p outside [0, 1]
        x = torch.zeros(B, T, 40, device=DEV)
        blob = torch.zeros(lib.ttrnn_rnn_param_count(C.byref(desc)), device=DEV)
        out = torch.empty(B, T, 256, device=DEV)
        sc = torch.empty(max(a.fwd_scratch_bytes, b.fwd_scratch_bytes) // 4 + 1, device=DEV)
        s = torch.cuda.current_stream().cuda_stream
        args = lambda ws: (C.byref(desc), C.byref(ws), x.data_ptr(), None, None, blob.data_ptr(), out.data_ptr(), None,
                           None, None, sc.data_ptr(), s)
        if L > 1:
            assert lib.ttrnn_rnn_forward(*args(b)) != 0 and b"TTRNN_WS_DROPOUT" in lib.ttrnn_last_error()
            assert lib.ttrnn_rnn_forward_dropout(*args(a), C.byref(_lib.Dropout(0.5, 0, 1, 0))) != 0
        for bad in (-0.1, 1.5, float("nan")):
            assert lib.ttrnn_rnn_forward_dropout(*args(b), C.byref(_lib.Dropout(bad, 0, 1, 0))) != 0
        assert lib.ttrnn_rnn_forward_dropout(*args(b), None) != 0
        torch.cuda.synchronize()


# ---- 3. mask properties -------------------------------------------------------------------------------------------
def test_keep_fraction_paths_and_global_rows():
    lib = _lib.load()
    s = torch.cuda.current_stream().cuda_stream
    for p in (0.1, 0.5, 0.9):
        dp = _lib.Dropout(p, 0, 1234, 8)
        B, T, F = 1000, 100, 128                         # 1.28e7 elements
        ones = torch.ones(B, T, F, device=DEV)
        y = torch.empty_like(ones)
        _lib.check(lib.ttrnn_dropout_apply(B, T, F, 0, 1, 0, C.byref(dp), ones.data_ptr(), y.data_ptr(), None, s), "apply")
        n = y.numel()
        frac = float((y != 0).double().mean())
        sigma = ((1 - p) * p / n) ** 0.5
        assert abs(frac - (1 - p)) <= 5 * sigma, (p, frac)
        # the scale is 1 / (1 - p) of the FP32 p the struct carries, rounded to FP32
        p32 = float(torch.tensor(p, dtype=torch.float32))
        assert torch.all((y == 0) | (y == float(torch.tensor(1.0 / (1.0 - p32), dtype=torch.float32))))
        # the scalar path (an unaligned pointer) draws the same mask as the float4 path
        buf = torch.ones(B * T * F + 1, device=DEV)
        y1 = torch.empty(B * T * F + 1, device=DEV)
        _lib.check(lib.ttrnn_dropout_apply(B, T, F, 0, 1, 0, C.byref(dp), buf[1:].data_ptr(), y1[1:].data_ptr(), None, s),
                   "apply")
        assert torch.equal(y1[1:].view(B, T, F), y)
        # rows 300 .. 599 on their own, with row0 = 300, are the same rows of the whole-batch mask; the reversed copy
        yr = torch.empty(300, T, F, device=DEV)
        ys = torch.empty(300, T, F, device=DEV)
        _lib.check(lib.ttrnn_dropout_apply(300, T, F, 300, 1, 0, C.byref(dp), ones[:300].data_ptr(), ys.data_ptr(),
                                           yr.data_ptr(), s), "apply")
        assert torch.equal(ys, y[300:600]) and torch.equal(yr, ys.flip(1))
        # another boundary, another offset: other masks
        for other in (_lib.Dropout(p, 0, 1234, 12), ):
            _lib.check(lib.ttrnn_dropout_apply(300, T, F, 300, 1, 0, C.byref(other), ones[:300].data_ptr(), ys.data_ptr(),
                                               None, s), "apply")
            assert not torch.equal(ys, y[300:600])
        _lib.check(lib.ttrnn_dropout_apply(300, T, F, 300, 0, 0, C.byref(dp), ones[:300].data_ptr(), ys.data_ptr(), None, s),
                   "apply")
        assert not torch.equal(ys, y[300:600])
    # backward: (dy + reverse(dy_rev)) * mask / (1 - p), in place
    dp = _lib.Dropout(0.3, 0, 99, 4)
    g = torch.randn(6, 7, 12, device=DEV)
    gr = torch.randn(6, 7, 12, device=DEV)
    mask = torch.empty_like(g)
    _lib.check(lib.ttrnn_dropout_apply(6, 7, 12, 2, 3, 0, C.byref(dp), torch.ones_like(g).data_ptr(), mask.data_ptr(), None,
                                       s), "apply")
    want = (g + gr.flip(1)) * mask
    _lib.check(lib.ttrnn_dropout_apply(6, 7, 12, 2, 3, 1, C.byref(dp), g.data_ptr(), g.data_ptr(), gr.data_ptr(), s), "apply")
    torch.cuda.synchronize()
    assert torch.equal(g, want)


@pytest.mark.parametrize("name", ["TTLSTM", "LSTM", "TTGRU_bidir"])
def test_seed_offset_successive_calls_and_no_grad(name):
    torch.manual_seed(3)
    if name == "TTLSTM":
        m = quiet(tr.TTLSTM, 40, 256, 3, torch.device("cpu"), n_cores=3, tt_rank=8, dropout=P)
    elif name == "LSTM":
        m = quiet(tr.LSTM, 128, 128, 3, torch.device("cpu"), dropout=P)
    else:
        m = quiet(tr.TTGRU, 16, 256, 2, torch.device("cpu"), n_cores=2, tt_rank=4, bidirectional=True, dropout=P)
    m = m.to(DEV)
    x = torch.rand(16, 9, m.input_size, device=DEV)

    def step():
        for q in m.parameters():
            q.grad = None
        xs = x.clone().requires_grad_(True)
        out = m(xs)[0]
        (out * out).sum().backward()
        torch.cuda.synchronize()
        return out.detach(), xs.grad, [q.grad.clone() for q in m.parameters()]

    torch.cuda.manual_seed(21)
    off0 = gen().get_offset()
    a = step()
    assert gen().get_offset() == off0 + 4
    b = step()
    assert gen().get_offset() == off0 + 8
    assert not torch.equal(a[0], b[0])                   # successive calls draw different masks
    torch.cuda.manual_seed(21)
    c = step()
    assert torch.equal(a[0], c[0]) and torch.equal(a[1], c[1]) and all(torch.equal(u, v) for u, v in zip(a[2], c[2]))
    # no_grad in training mode masks with the same draw as the training forward
    gen().set_offset(off0)
    with torch.no_grad():
        d = m(x)[0]
    assert torch.equal(d, a[0])
    # eval mode: no mask, no draw, the module without dropout
    m.eval()
    off = gen().get_offset()
    e = m(x)[0]
    m.dropout = 0.0
    f = m(x)[0]
    assert gen().get_offset() == off and torch.equal(e, f)


def test_dropout_under_stream_capture_raises():
    m = quiet(tr.TTLSTM, 40, 256, 2, torch.device("cpu"), n_cores=3, tt_rank=8, dropout=P).to(DEV)
    x = torch.rand(8, 4, 40, device=DEV)
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with pytest.raises(RuntimeError, match="graph-safe"):
            with torch.cuda.graph(g, stream=s):
                with torch.no_grad():
                    m(x)
    torch.cuda.synchronize()


# ---- 4. p = 1 -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cell", ["lstm", "gru"])
def test_p_one_is_finite_with_zero_upper_ih_gradients(cell):
    L, H = 3, 256
    cls = tr.TTLSTM if cell == "lstm" else tr.TTGRU
    m = quiet(cls, 40, H, L, torch.device("cpu"), n_cores=3 if cell == "lstm" else 2, tt_rank=8 if cell == "lstm" else 4,
              dropout=1.0).to(DEV)
    x = torch.rand(24, 8, 40, device=DEV, requires_grad=True)
    out, fin = m.forward_states(x)
    h = fin[0] if cell == "lstm" else fin
    # the output no longer depends on layer 0; every layer's final state does on its own layer
    ((out * out).sum() + h.sum()).backward()
    torch.cuda.synchronize()
    assert torch.isfinite(out).all() and torch.isfinite(h).all() and torch.isfinite(x.grad).all()
    assert torch.count_nonzero(x.grad) > 0
    for l in range(L):
        cell_l = getattr(m, "cell%d" % l)
        for q in cell_l.parameters():
            assert torch.isfinite(q.grad).all()
        cores = list(cell_l.input_weights.weight_t.tt_cores)
        if l > 0:
            assert all(torch.count_nonzero(c.grad) == 0 for c in cores), l
        else:
            assert any(torch.count_nonzero(c.grad) > 0 for c in cores)


# ---- 5. other modules ---------------------------------------------------------------------------------------------
OTHER = [
    # name, kind, cell, I, H, L, d, r, B, T, bidirectional
    ("ttlstm_cfg3_bidir_L3", "tt", "lstm", 40, 256, 3, 3, 8, 12, 5, True),
    ("ttgru_bidir_L2", "tt", "gru", 16, 256, 2, 2, 4, 12, 6, True),
    ("dense_lstm_bidir_L2", "dense", "lstm", 128, 128, 2, 0, 0, 8, 6, True),
    ("dense_gru_bidir_L3", "dense", "gru", 128, 128, 3, 0, 0, 8, 5, True),
    ("dense_lstm_L3", "dense", "lstm", 128, 128, 3, 0, 0, 8, 6, False),
    ("dense_gru_L2", "dense", "gru", 128, 256, 2, 0, 0, 10, 7, False),
]
CLS = {("tt", "lstm"): tr.TTLSTM, ("tt", "gru"): tr.TTGRU, ("dense", "lstm"): tr.LSTM, ("dense", "gru"): tr.GRU}


@pytest.mark.parametrize("case", OTHER, ids=[c[0] for c in OTHER])
def test_other_modules_match_reference_composition(case):
    name, kind, cell, I, H, L, d, r, B, T, bidir = case
    D = 2 if bidir else 1
    torch.manual_seed(11)
    kw = dict(n_cores=d, tt_rank=r) if kind == "tt" else {}
    m = quiet(CLS[(kind, cell)], I, H, L, torch.device("cpu"), bidirectional=bidir, dropout=P, **kw)
    g = torch.Generator().manual_seed(7)
    x = torch.rand(B, T, I, generator=g)
    st = [0.5 * torch.randn(D * L, B, H, generator=g) for _ in range(2 if cell == "lstm" else 1)]
    w = [torch.randn(B, T, D * H, generator=g)] + [torch.randn(D * L, B, H, generator=g) for _ in st]
    # the engine's run
    md = m.to(DEV)
    for q in md.parameters():
        q.grad = None
    xs = x.clone().to(DEV).requires_grad_(True)
    ss = [s.clone().to(DEV).requires_grad_(True) for s in st]
    seed, offset = draw_state()
    out, fin = md.forward_states(xs, tuple(ss) if cell == "lstm" else ss[0])
    fin = list(fin) if cell == "lstm" else [fin]
    loss = (out * w[0].to(DEV)).sum() + sum((f * wf.to(DEV)).sum() for f, wf in zip(fin, w[1:]))
    loss.backward()
    torch.cuda.synchronize()
    assert gen().get_offset() == offset + 4
    got_dp = [q.grad for q in md.flat_parameters()]
    masks = [mk.double().cpu() for mk in engine_masks(P, seed, offset, L, B, T, D * H)]
    # the reference composition
    sd = {k: v.detach().double().cpu() for k, v in md.state_dict().items()}
    if kind == "tt":
        fwd = oracle.lstm_forward if cell == "lstm" else oracle.gru_forward
        lay = lambda s, n: oracle.layers_from_state_dict(s, n, dtype=torch.float64, requires_grad=True)
        flat = oracle.flat_params
    else:
        fwd = dense_oracle.lstm_forward if cell == "lstm" else dense_oracle.gru_forward
        lay = lambda s, n: dense_oracle.layers_from_state_dict(s, n, requires_grad=True)
        flat = dense_oracle.flat_params
    xr = x.double().requires_grad_(True)
    sr = [s.double().requires_grad_(True) for s in st]
    if bidir:
        pairs = bidir_layers(lambda s, n, **k: lay(s, n), sd, L)
        o_ref, f_ref = dropout_bidir_forward(fwd, cell, pairs, xr, masks, sr)
        params = flat(flat_pairs(pairs))
    else:
        layers = lay(sd, L)
        o_ref, f_ref = dropout_layer_states(fwd, cell, layers, xr, masks, sr)
        params = flat(layers)
    ((o_ref * w[0].double()).sum() + sum((f * wf.double()).sum() for f, wf in zip(f_ref, w[1:]))).backward()
    assert rel_err(out, o_ref) <= FWD_TOL, rel_err(out, o_ref)
    for a, b in zip(fin, f_ref):
        for i in range(D * L):
            assert rel_err(a[i], b[i]) <= FWD_TOL, (i, rel_err(a[i], b[i]))
    assert rel_err(xs.grad, xr.grad) <= GRAD_TOL, rel_err(xs.grad, xr.grad)
    for a, b in zip(ss, sr):
        for i in range(D * L):
            assert rel_err(a.grad[i], b.grad[i]) <= GRAD_TOL, (i, rel_err(a.grad[i], b.grad[i]))
    assert len(got_dp) == len(params)
    for i, (a, b) in enumerate(zip(got_dp, params)):
        assert rel_err(a, b.grad) <= GRAD_TOL, (i, tuple(b.shape), rel_err(a, b.grad))
