"""Variable-length rows (DESIGN.md §4.22) on the GPU.

The engine's padded call with per-row lengths (a PackedSequence through the modules) against
  - per-row fixed-length calls of the same module on x[b:b+1, :len_b] (every route, per-layer states, gradients of the
    input, the states and every parameter), and
  - the FP64 references of tests/varlen_ref.py (the oracle row by row, torch.nn.LSTM / GRU on a PackedSequence).
Also: zero padding of outputs and input gradients, lengths all equal to T against the call without lengths, no_grad and
repeat bit-identity, large finite padded inputs, bidirectional stacks, dropout, the static route, rank-one I = 1, and
SpeakerEncoder.embed_utterances(using_partials=False).  Bars: 1e-5 forward, 1e-4 gradients (norm-wise relative).
"""
import ctypes
import io
from contextlib import redirect_stdout

import numpy as np
import pytest
import torch
from torch.nn.utils.rnn import pack_padded_sequence, pad_packed_sequence

import tensorized_rnn_b200 as tr
from tensorized_rnn_b200 import _lib
from tensorized_rnn_b200.functional import rnn_sequence
from helpers import FWD_TOL, GRAD_TOL, oracle, rel_err
from varlen_ref import oracle_rows, torch_packed

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
CPU = torch.device("cpu")
C_i64 = ctypes.c_int64


def make(kind, cell, I, H, L, seed=5, **kw):
    torch.manual_seed(seed)
    if kind == "dense":
        cls = tr.LSTM if cell == "lstm" else tr.GRU
        return cls(I, H, L, CPU, **kw).to(DEV)
    d, r = kind
    cls = tr.TTLSTM if cell == "lstm" else tr.TTGRU
    return cls(I, H, L, CPU, n_cores=d, tt_rank=r, **kw).to(DEV)


def n_states(m):
    return 2 if m.cell_kind == "lstm" else 1


def widths(m):
    return [m.output_size, m.hidden_size][:n_states(m)]


def unpack(res, T):
    out, st = res
    out = pad_packed_sequence(out, batch_first=True, total_length=T)[0]
    return out, list(st) if isinstance(st, tuple) else [st]


def run_packed(m, x, lengths, states):
    packed = pack_padded_sequence(x, torch.as_tensor(lengths), batch_first=True, enforce_sorted=False)
    st = None if states is None else (tuple(states) if len(states) > 1 else states[0])
    return unpack(m.forward_states(packed, st), x.shape[1])


def run_rows(m, x, lengths, states):
    """Per-row fixed-length calls, stitched into the padded contract."""
    B, T, _ = x.shape
    outs, fins = [], []
    for b, n in enumerate(lengths):
        st = None if states is None else tuple(s[:, b:b + 1] for s in states)
        o, f = m.forward_states(x[b:b + 1, :n], st if st is None or len(st) > 1 else st[0])
        outs.append(torch.cat([o, o.new_zeros(1, T - n, o.shape[2])], dim=1))
        fins.append(list(f) if isinstance(f, tuple) else [f])
    return torch.cat(outs), [torch.cat([f[k] for f in fins], dim=1) for k in range(len(fins[0]))]


def data(m, B, T, lengths, seed=9, init=True):
    g = torch.Generator().manual_seed(seed)
    D = 2 if m.bidirectional else 1
    x = torch.rand(B, T, m.input_size, generator=g) - 0.5
    x = x * (torch.arange(T)[None, :, None] < torch.as_tensor(lengths)[:, None, None])
    st = [0.5 * torch.randn(D * m.num_layers, B, w, generator=g) for w in widths(m)] if init else None
    w = [torch.randn(B, T, D * m.output_size, generator=g)] + [torch.randn(D * m.num_layers, B, wd, generator=g)
                                                                for wd in widths(m)]
    to = lambda t: t.to(DEV).requires_grad_()
    return to(x), (None if st is None else [to(s) for s in st]), [t.to(DEV) for t in w]


def grads_of(m, x, st, w, fn, lengths):
    out, fin = fn(m, x, lengths, st)
    loss = (out * w[0]).sum() + sum((f * wk).sum() for f, wk in zip(fin, w[1:]))
    inputs = [x] + ([] if st is None else st) + list(m.parameters())
    g = torch.autograd.grad(loss, inputs, allow_unused=True)
    return out.detach(), [f.detach() for f in fin], g


def check_against_rows(m, B, T, lengths, init=True):
    x, st, w = data(m, B, T, lengths, init=init)
    out, fin, g = grads_of(m, x, st, w, run_packed, lengths)
    out_r, fin_r, g_r = grads_of(m, x, st, w, run_rows, lengths)
    pad = torch.arange(T, device=DEV)[None, :] >= torch.as_tensor(lengths, device=DEV)[:, None]
    assert (out[pad] == 0).all()
    assert rel_err(out, out_r) <= FWD_TOL, rel_err(out, out_r)
    for a, b in zip(fin, fin_r):
        assert rel_err(a, b) <= FWD_TOL, rel_err(a, b)
    assert (g[0][pad] == 0).all()
    names = ["x"] + ["state%d" % k for k in range(0 if st is None else len(st))] + [n for n, _ in m.named_parameters()]
    bad = {n: rel_err(a, b) for n, a, b in zip(names, g, g_r) if a is not None and not rel_err(a, b) <= GRAD_TOL}
    assert not bad, bad
    return out, fin


LENGTHS = [7, 1, 12, 4, 12, 9, 2]          # 1 and T, unsorted, repeats
CASES = [
    # name, kind, cell, I, H, L, kwargs
    ("tt_lstm_d2r4_L1", (2, 4), "lstm", 16, 64, 1, {}),
    ("tt_lstm_d2r4_L2", (2, 4), "lstm", 16, 64, 2, {}),
    ("tt_lstm_d2r4_L3_nobias", (2, 4), "lstm", 16, 64, 3, dict(bias=False)),
    ("tt_gru_d2r4_L2", (2, 4), "gru", 16, 64, 2, {}),
    ("tt_gru_d2r4_L3_nobias", (2, 4), "gru", 16, 64, 3, dict(bias=False)),
    ("tt_lstm_d3r8_L2", (3, 8), "lstm", 40, 256, 2, {}),
    ("tt_gru_d3r8_L1", (3, 8), "gru", 40, 256, 1, {}),
    ("tt_lstm_I1_L2", (2, 4), "lstm", 1, 64, 2, {}),
    ("tt_gru_I1_L1", (2, 4), "gru", 1, 64, 1, {}),
    ("tt_lstm_proj_L2", (2, 4), "lstm", 16, 64, 2, dict(proj_size=16)),
    ("dense_lstm_L2", "dense", "lstm", 128, 128, 2, {}),
    ("dense_gru_L3_nobias", "dense", "gru", 128, 128, 3, dict(bias=False)),
    ("dense_lstm_proj_L2", "dense", "lstm", 128, 256, 2, dict(proj_size=128)),
]


@pytest.mark.parametrize("name,kind,cell,I,H,L,kw", CASES, ids=[c[0] for c in CASES])
def test_against_per_row_calls(name, kind, cell, I, H, L, kw):
    check_against_rows(make(kind, cell, I, H, L, **kw), len(LENGTHS), 12, LENGTHS)


@pytest.mark.parametrize("chunk,static", [(4, 1), (5, 0), (0, 0)])
def test_chunks_and_runtime_kernels(chunk, static):
    lib = _lib.load()
    lib.ttrnn_set_option(b"chunk_steps", chunk)
    lib.ttrnn_set_option(b"static_kernels", static)
    try:
        for cell in ("lstm", "gru"):
            check_against_rows(make((2, 4), cell, 16, 64, 2), len(LENGTHS), 12, LENGTHS)
    finally:
        lib.ttrnn_set_option(b"chunk_steps", 0)
        lib.ttrnn_set_option(b"static_kernels", 1)


def row_groups_of(m, B, T):
    """Row groups of the lengths plan the call at (B, T) runs (ttrnn_rnn_describe_ex)."""
    return _lib.describe_plan(m.spec().desc(B, T), training=True,
                              flags=_lib.WS_LENGTHS | _lib.WS_LAYER_STATES)[0]["row_groups"]


def test_planned_row_groups_static_route_full_gradients():
    """The cfg3 stack at its batch (B 640): several CTA waves, the planned two row groups (the second group runs from
    lengths + its first row), the static kernels (launch counters); outputs, every final state and the gradients of x,
    the states and every parameter against per-row calls."""
    lib = _lib.load()
    m = make((3, 8), "lstm", 40, 256, 3)
    B, T = 640, 9
    assert row_groups_of(m, B, T) == 2
    lengths = ((np.arange(B) * 7) % T + 1).tolist()
    lib.ttrnn_static_kernel_launches(None, 0, 1)
    check_against_rows(m, B, T, lengths)
    counts = (C_i64 * 4096)()
    n = lib.ttrnn_static_kernel_launches(counts, 4096, 1)
    assert sum(counts[:n]) > 0


@pytest.mark.parametrize("cell", ["lstm", "gru"])
def test_forced_row_groups(cell):
    """A small batch cut into two row groups (group 0 = 12 rows) with lengths 1 and T on both sides of the cut."""
    lib = _lib.load()
    lib.ttrnn_set_option(b"row_groups", 12)
    try:
        m = make((2, 4), cell, 16, 64, 2)
        lengths = LENGTHS + LENGTHS[::-1] + [12, 1, 5, 8, 3, 12]
        assert row_groups_of(m, len(lengths), 12) == 2
        check_against_rows(m, len(lengths), 12, lengths)
    finally:
        lib.ttrnn_set_option(b"row_groups", 1)


def test_describe_reports_the_route_under_lengths():
    """I = 1: without lengths layer 0 takes the rank-one input mode, with them the materialised projection."""
    m = make((2, 4), "lstm", 1, 64, 2)
    desc = m.spec().desc(8, 12)
    assert _lib.describe_plan(desc)[1]["ih_route"] == "rank_one"
    assert _lib.describe_plan(desc, flags=_lib.WS_LENGTHS)[1]["ih_route"] != "rank_one"


@pytest.mark.parametrize("cell", ["lstm", "gru"])
def test_fp64_references(cell):
    """The shared-state forward() against the oracle row by row and torch's PackedSequence path, FP64."""
    m = make((2, 4), cell, 16, 64, 2)
    layers = oracle.layers_from_state_dict({k: v.detach().cpu().double() for k, v in m.state_dict().items()}, 2)
    g = torch.Generator().manual_seed(2)
    x = torch.rand(len(LENGTHS), 12, 16, generator=g, dtype=torch.float64)
    h0 = [0.5 * torch.randn(len(LENGTHS), 64, generator=g, dtype=torch.float64) for _ in range(n_states(m))]
    packed = pack_padded_sequence(x.float().to(DEV), torch.as_tensor(LENGTHS), batch_first=True, enforce_sorted=False)
    out, st = m(packed, tuple(h.float().to(DEV) for h in h0) if cell == "lstm" else h0[0].float().to(DEV))
    out = pad_packed_sequence(out, batch_first=True, total_length=12)[0]
    st = list(st) if cell == "lstm" else [st]
    ref_init = tuple(h0) if cell == "lstm" else h0[0]
    for ref in (oracle_rows(cell, layers, x, LENGTHS, ref_init), torch_packed(cell, layers, x, LENGTHS, ref_init)):
        assert rel_err(out, ref[0]) <= FWD_TOL
        for a, b in zip(st, ref[1:]):
            assert rel_err(a, b) <= FWD_TOL


@pytest.mark.parametrize("kind,cell,I,H,kw", [((2, 4), "lstm", 16, 64, {}), ((2, 4), "gru", 16, 64, {}),
                                             ("dense", "lstm", 128, 128, {}), ("dense", "gru", 128, 128, {})])
def test_bidirectional(kind, cell, I, H, kw):
    check_against_rows(make(kind, cell, I, H, 2, bidirectional=True, **kw), len(LENGTHS), 12, LENGTHS)


@pytest.mark.parametrize("kind,cell,I,H", [((2, 4), "lstm", 16, 64), ((3, 8), "lstm", 40, 256), ((2, 4), "gru", 16, 64),
                                          ("dense", "lstm", 128, 128), ("dense", "gru", 128, 128)])
def test_all_lengths_T_matches_the_call_without_lengths(kind, cell, I, H):
    m = make(kind, cell, I, H, 2)
    B, T = 9, 10
    lengths = [T] * B
    x, st, w = data(m, B, T, lengths)
    out, fin, g = grads_of(m, x, st, w, run_packed, lengths)

    def plain(m_, x_, lengths_, st_):
        o, f = m_.forward_states(x_, tuple(st_) if len(st_) > 1 else st_[0])
        return o, list(f) if isinstance(f, tuple) else [f]

    out0, fin0, g0 = grads_of(m, x, st, w, plain, lengths)
    assert torch.equal(out, out0)
    for a, b in zip(fin, fin0):
        assert torch.equal(a, b)
    for a, b in zip(g, g0):
        if a is not None:
            assert rel_err(a, b) <= GRAD_TOL


@pytest.mark.parametrize("kind,cell,I,H", [((2, 4), "lstm", 16, 64), ((2, 4), "gru", 16, 64), ("dense", "lstm", 128, 128)])
def test_no_grad_repeat_and_padding_values(kind, cell, I, H):
    m = make(kind, cell, I, H, 2)
    x, st, _ = data(m, len(LENGTHS), 12, LENGTHS)
    a = run_packed(m, x, LENGTHS, st)
    b = run_packed(m, x, LENGTHS, st)
    with torch.no_grad():
        c = run_packed(m, x, LENGTHS, st)
    for u, v, z in zip([a[0]] + a[1], [b[0]] + b[1], [c[0]] + c[1]):
        assert torch.equal(u, v) and torch.equal(u, z)
    # the padded form with large finite values past each length gives the same results and parameter gradients
    pad = torch.arange(12, device=DEV)[None, :, None] >= torch.as_tensor(LENGTHS, device=DEV)[:, None, None]
    results = []
    for fill in (0.0, 1e6):
        xx = torch.where(pad, torch.full_like(x, fill), x.detach())
        m.zero_grad(set_to_none=True)
        out, (h, *rest) = _padded(m, xx, LENGTHS, st)
        (out.sum() + h.sum()).backward()
        results.append([out.detach(), h.detach()] + [p.grad.clone() for p in m.parameters()])
    for u, v in zip(*results):
        assert torch.equal(u, v)


def _padded(m, x, lengths, st):
    """The engine-native padded form: rnn_sequence / the dense function with lengths."""
    if isinstance(m, (tr.TTLSTM, tr.TTGRU)):
        res = rnn_sequence(m.spec(), x, *(s.detach() for s in st), *([None] if len(st) == 1 else []), m.flat_parameters(),
                           layer_states=True, lengths=lengths)
        return res[0], res[1:]
    res = m._run_padded(x, *(s.detach() for s in st), *([None] if len(st) == 1 else []), True, lengths)
    return res[0], res[1:]


@pytest.mark.parametrize("kind,cell,I,H", [((2, 4), "lstm", 16, 64), ("dense", "gru", 128, 128)])
def test_dropout(kind, cell, I, H):
    """p = 0.3 with the engine's mask: lengths all T reproduce the call without lengths under the same draw; with
    varied lengths the padding stays zero and two draws from one seed agree."""
    m = make(kind, cell, I, H, 3, dropout=0.3).train()
    B, T = 8, 10
    full = [T] * B
    x, st, _ = data(m, B, T, full)
    torch.cuda.manual_seed(3)
    a = run_packed(m, x, full, st)
    torch.cuda.manual_seed(3)
    b = m.forward_states(x, tuple(st) if len(st) > 1 else st[0])
    assert torch.equal(a[0], b[0])
    lengths = [10, 3, 1, 7, 10, 5, 2, 9]
    torch.cuda.manual_seed(4)
    c = run_packed(m, x, lengths, st)
    torch.cuda.manual_seed(4)
    d = run_packed(m, x, lengths, st)
    pad = torch.arange(T, device=DEV)[None, :] >= torch.as_tensor(lengths, device=DEV)[:, None]
    assert (c[0][pad] == 0).all() and torch.equal(c[0], d[0])
    c[0].sum().backward()
    assert (x.grad[pad] == 0).all()


@pytest.mark.parametrize("kind,cell,I,H", [((2, 4), "lstm", 16, 64), ("dense", "gru", 128, 128)])
def test_bidirectional_dropout(kind, cell, I, H):
    """Bidirectional L = 2 with p = 0.3: the joined output is masked, then reversed over each row's length.  Lengths all T
    reproduce the call without lengths under the same draw, outputs and final states bit for bit; with varied lengths the
    padding and its input gradient stay zero and two calls from one seed agree."""
    m = make(kind, cell, I, H, 2, bidirectional=True, dropout=0.3).train()
    B, T = 8, 10
    full = [T] * B
    x, st, _ = data(m, B, T, full)
    torch.cuda.manual_seed(3)
    a = run_packed(m, x, full, st)
    torch.cuda.manual_seed(3)
    b = m.forward_states(x, tuple(st) if len(st) > 1 else st[0])
    assert torch.equal(a[0], b[0])
    bf = list(b[1]) if isinstance(b[1], tuple) else [b[1]]
    for u, v in zip(a[1], bf):
        assert torch.equal(u, v)
    lengths = [10, 3, 1, 7, 10, 5, 2, 9]
    torch.cuda.manual_seed(4)
    c = run_packed(m, x, lengths, st)
    torch.cuda.manual_seed(4)
    d = run_packed(m, x, lengths, st)
    pad = torch.arange(T, device=DEV)[None, :] >= torch.as_tensor(lengths, device=DEV)[:, None]
    assert (c[0][pad] == 0).all() and torch.equal(c[0], d[0])
    (c[0].sum() + sum(f.sum() for f in c[1])).backward()
    assert (x.grad[pad] == 0).all() and torch.isfinite(x.grad).all()


# ---- SpeakerEncoder full-utterance mode ---------------------------------------------------------------------------------
ENC = {"spkenc_tt_lstm_h64_L2": dict(compression="tt", n_cores=3, rank=4),
       "spkenc_dense_lstm_h128_L1": dict(compression=None),
       "spkenc_tt_gru_h64_L1": dict(compression="tt", n_cores=2, rank=2, use_gru=True)}
PROJ = {"proj_tt_lstm_h64_p16_L2": (64, 2, dict(compression="tt", n_cores=2, rank=4, proj_size=16)),
        "proj_dense_lstm_h256_p128_L1": (256, 1, dict(compression=None, proj_size=128))}


def _encoder(name):
    import os
    from helpers import GOLDEN
    if name in PROJ:
        H, L, kw = PROJ[name]
        torch.manual_seed(6)
        with redirect_stdout(io.StringIO()):
            enc = tr.SpeakerEncoder(40, H, L, 32, CPU, None, **kw)
        return enc.to(DEV)
    g = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    _, _, _, H, L = (int(v) for v in g["shape"])
    with redirect_stdout(io.StringIO()):
        enc = tr.SpeakerEncoder(40, H, L, 32, CPU, None, **ENC[name])
    enc.load_state_dict({k[len("param:"):]: torch.from_numpy(v) for k, v in g.items() if k.startswith("param:")})
    return enc.to(DEV)


@pytest.mark.parametrize("name", sorted(ENC) + sorted(PROJ))
def test_embed_utterances_full_mode(name):
    enc = _encoder(name)
    lengths = [1, 3000, 160, 57, 999, 2]
    frames = torch.rand(sum(lengths), 40, generator=torch.Generator().manual_seed(7)).to(DEV)
    w = torch.randn(len(lengths), 32, generator=torch.Generator().manual_seed(8)).to(DEV)
    d = enc.embed_utterances(frames, lengths, using_partials=False)
    assert d.shape == (len(lengths), 32)
    (d * w).sum().backward()
    grads = {k: p.grad.clone() for k, p in enc.named_parameters() if p.grad is not None}
    enc.zero_grad(set_to_none=True)
    ref = torch.cat([enc(u[None]) for u in torch.split(frames, lengths)])
    assert rel_err(d, ref) <= FWD_TOL, rel_err(d, ref)
    (ref * w).sum().backward()
    ref_grads = {k: p.grad for k, p in enc.named_parameters() if p.grad is not None}
    assert set(grads) == set(ref_grads) == {k for k, _ in enc.named_parameters() if not k.startswith("similarity_")}
    bad = {k: rel_err(grads[k], ref_grads[k]) for k in grads if not rel_err(grads[k], ref_grads[k]) <= GRAD_TOL}
    assert not bad, bad
