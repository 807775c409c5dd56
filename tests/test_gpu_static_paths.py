"""GPU parity of the statically specialised kernels at the benchmark shapes (BASELINE.json configs 1-5).

The reference fixtures use tiny batches, which (by design) exercise the runtime-shape kernels for the
batched ih projection; these tests use enough rows (B*T >= 64) and enough batch rows to reach every
static kernel: recurrent forward/backward (all five hh shapes), rank-one input mode, batched TT matvec
forward/backward, multi-chunk execution, ragged last batch tile.  The oracle (CPU restatement of the
reference, pinned by tests/test_oracle.py) provides the expected values on the same seeded inputs.
Tolerances: 1e-5 forward, 1e-4 gradients (north_star), norm-wise relative.
"""
import ctypes

import pytest
import torch

import tensorized_rnn_b200 as tr
from tensorized_rnn_b200 import _lib
from helpers import FWD_TOL, GRAD_TOL, oracle, quiet, rel_err

pytestmark = pytest.mark.gpu

# name, cell, I, H, L, d, r, B, T, with_init, chunk_steps
CASES = [
    ("cfg1_shape", "lstm", 1, 256, 1, 2, 4, 9, 12, False, 0),
    ("cfg2_shape", "gru", 1, 256, 1, 2, 4, 17, 10, True, 0),
    ("cfg2_shape_chunked", "gru", 1, 256, 1, 2, 4, 6, 9, False, 4),
    ("cfg3_shape", "lstm", 40, 256, 3, 3, 8, 13, 8, True, 0),
    ("cfg3_shape_chunked", "lstm", 40, 256, 3, 3, 8, 10, 9, False, 4),
    ("cfg4_shape", "lstm", 40, 256, 3, 4, 16, 5, 14, False, 0),
    ("cfg5_shape", "lstm", 256, 1024, 1, 4, 8, 4, 17, True, 0),
    ("cfg1_shape_xgrad", "lstm", 1, 256, 1, 2, 4, 8, 9, False, 0),     # x.requires_grad: XG-mode kernels
    # row-by-row MNIST (pmnist_test.py without --permute: I = 28, T = 28): ih shape with no static chain kernel
    # (dense route forward, chain route backward because dX is requested), XG-mode kept-gates BPTT kernels
    ("rowmnist_lstm", "lstm", 28, 256, 1, 2, 4, 12, 28, False, 0),
    ("rowmnist_gru_L2", "gru", 28, 256, 2, 2, 4, 9, 28, True, 0),
]


def _sd_from_layers(layers):
    sd = {}
    for li, p in enumerate(layers):
        for short, long in (("ih", "input_weights"), ("hh", "hidden_weights")):
            for k, c in enumerate(p[short + "_cores"]):
                sd["cell%d.%s.parameters.%d" % (li, long, k)] = c.detach().clone()
            if p[short + "_bias"] is not None:
                sd["cell%d.%s.bias" % (li, long)] = p[short + "_bias"].detach().clone()
    return sd


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_static_kernels_match_oracle(case):
    name, cell, I, H, L, d, r, B, T, with_init, chunk = case
    dev = torch.device("cuda:0")
    lib = _lib.load()
    layers = oracle.random_layers(cell, I, H, L, d, r, bias=True, seed=123, requires_grad=True, scale=1.5)
    g = torch.Generator().manual_seed(77)
    x = torch.rand(B, T, I, generator=g)
    want_dx = name.endswith("xgrad") or I > 1
    x_ref = x.clone().requires_grad_(want_dx)
    init_ref = None
    if with_init:
        h0 = (0.3 * torch.randn(B, H, generator=g)).requires_grad_(True)
        init_ref = (h0, (0.3 * torch.randn(B, H, generator=g)).requires_grad_(True)) if cell == "lstm" else h0
    w_out = torch.randn(B, T, H, generator=g)
    w_h = torch.randn(B, H, generator=g)
    if cell == "lstm":
        o_ref, (h_ref, c_ref) = oracle.lstm_forward(layers, x_ref, init_ref)
        loss = (o_ref * w_out).sum() + (h_ref * w_h).sum() + (c_ref * w_h).sum()
    else:
        o_ref, h_ref = oracle.gru_forward(layers, x_ref, init_ref)
        loss = (o_ref * w_out).sum() + (h_ref * w_h).sum()
    loss.backward()

    cls = tr.TTLSTM if cell == "lstm" else tr.TTGRU
    m = quiet(cls, I, H, L, torch.device("cpu"), n_cores=d, tt_rank=r)
    m.load_state_dict(_sd_from_layers(layers))
    m = m.to(dev)
    xd = x.to(dev).requires_grad_(want_dx)
    init = None
    if with_init:
        h0d = init_ref[0].detach().to(dev).requires_grad_(True) if cell == "lstm" else init_ref.detach().to(dev).requires_grad_(True)
        init = (h0d, init_ref[1].detach().to(dev).requires_grad_(True)) if cell == "lstm" else h0d
    lib.ttrnn_set_option(b"chunk_steps", chunk)
    try:
        if cell == "lstm":
            out, (h, c) = m(xd, init)
            loss = (out * w_out.to(dev)).sum() + (h * w_h.to(dev)).sum() + (c * w_h.to(dev)).sum()
        else:
            out, h = m(xd, init)
            loss = (out * w_out.to(dev)).sum() + (h * w_h.to(dev)).sum()
        loss.backward()
        torch.cuda.synchronize()
    finally:
        lib.ttrnn_set_option(b"chunk_steps", 0)
    assert rel_err(out, o_ref) <= FWD_TOL
    assert rel_err(h, h_ref) <= FWD_TOL
    if cell == "lstm":
        assert rel_err(c, c_ref) <= FWD_TOL
    errs = {}
    for p, ref in zip(m.flat_parameters(), oracle.flat_params(layers)):
        errs[tuple(p.shape)] = max(errs.get(tuple(p.shape), 0.0), rel_err(p.grad, ref.grad))
    if want_dx:
        errs["dx"] = rel_err(xd.grad, x_ref.grad)
    if with_init:
        if cell == "lstm":
            errs["dh0"] = rel_err(init[0].grad, init_ref[0].grad)
            errs["dc0"] = rel_err(init[1].grad, init_ref[1].grad)
        else:
            errs["dh0"] = rel_err(init.grad, init_ref.grad)
    bad = {k: v for k, v in errs.items() if not v <= GRAD_TOL}
    assert not bad, "gradient rel err above %.0e: %s" % (GRAD_TOL, bad)


def test_saved_activation_backward_matches_recompute():
    """Two backward variants of the static BPTT kernel must agree: full recompute (`save_u_bytes` 0) and kept
    gate activations (`save_u_bytes`, the default: backward skips the final stage of the recompute)."""
    dev = torch.device("cuda:0")
    lib = _lib.load()
    cases = [("gru", tr.TTGRU, 1, 256, 1, 2, 4), ("lstm", tr.TTLSTM, 1, 256, 1, 2, 4), ("lstm", tr.TTLSTM, 40, 256, 2, 3, 8)]
    for cell, cls, I, H, L, d, r in cases:
        torch.manual_seed(21)
        m = quiet(cls, I, H, L, torch.device("cpu"), n_cores=d, tt_rank=r).to(dev)
        x = torch.rand(19, 23, I, device=dev)
        res = []
        for save_u in (0, 1 << 30):
            lib.ttrnn_set_option(b"save_u_bytes", save_u)
            try:
                for p in m.parameters():
                    p.grad = None
                rr = m(x)
                out = rr[0]
                h = rr[1][0] if cell == "lstm" else rr[1]
                (out.sum() + 3 * h.sum()).backward()
                res.append((out.detach().clone(), [p.grad.clone() for p in m.parameters()]))
            finally:
                lib.ttrnn_set_option(b"save_u_bytes", 16 << 30)
        for other in res[1:]:
            assert torch.equal(res[0][0], other[0])
            for a, b in zip(res[0][1], other[1]):
                assert rel_err(b, a) <= GRAD_TOL


def test_dense_and_tt_chain_ih_routes_agree():
    """The batched ih projection contracted core by core (dense_ih = 0) and through the densified W_ih
    (dense_ih = 1, the default where it is cheaper) are the same map: outputs and every gradient must agree,
    including dX of inner layers and the TT-core gradients obtained by projecting the dense gradient."""
    dev = torch.device("cuda:0")
    lib = _lib.load()
    for cell, cls, I, H, L, d, r in (("lstm", tr.TTLSTM, 40, 256, 3, 3, 8), ("gru", tr.TTGRU, 28, 256, 2, 4, 16)):
        torch.manual_seed(33)
        m = quiet(cls, I, H, L, torch.device("cpu"), n_cores=d, tt_rank=r).to(dev)
        desc = m.spec().desc(11, 13)
        routes = [lib.ttrnn_rnn_ih_route(ctypes.byref(desc), l, None, None) for l in range(L)]
        assert all(rt == 1 for rt in routes), routes
        x = torch.rand(11, 13, I, device=dev)
        w = torch.randn(11, 13, H, device=dev)
        res = []
        for flag in (1, 0):
            lib.ttrnn_set_option(b"dense_ih", flag)
            try:
                for p in m.parameters():
                    p.grad = None
                rr = m(x)
                ((rr[0] * w).sum()).backward()
                res.append((rr[0].detach().clone(), [p.grad.clone() for p in m.parameters()]))
            finally:
                lib.ttrnn_set_option(b"dense_ih", 1)
        assert rel_err(res[0][0], res[1][0]) <= FWD_TOL
        for a, b in zip(res[0][1], res[1][1]):
            assert rel_err(a, b) <= GRAD_TOL


def test_dense_route_split_reduction_and_chunk_accumulation():
    """Dense ih route at a size that splits the X^T delta reduction over many CTAs and accumulates it over
    several time chunks (chunk_steps = 16 of T = 40), against the core-by-core route on the same inputs."""
    dev = torch.device("cuda:0")
    lib = _lib.load()
    torch.manual_seed(41)
    m = quiet(tr.TTLSTM, 40, 256, 2, torch.device("cpu"), n_cores=3, tt_rank=8).to(dev)
    x = torch.rand(64, 40, 40, device=dev, requires_grad=True)
    w = torch.randn(64, 40, 256, device=dev)
    res = []
    for dense, chunk in ((1, 16), (0, 0)):
        lib.ttrnn_set_option(b"dense_ih", dense)
        lib.ttrnn_set_option(b"chunk_steps", chunk)
        try:
            for p in m.parameters():
                p.grad = None
            x.grad = None
            out, (h, c) = m(x)
            ((out * w).sum() + c.sum()).backward()
            res.append((out.detach().clone(), x.grad.clone(), [p.grad.clone() for p in m.parameters()]))
        finally:
            lib.ttrnn_set_option(b"dense_ih", 1)
            lib.ttrnn_set_option(b"chunk_steps", 0)
    assert rel_err(res[0][0], res[1][0]) <= FWD_TOL
    assert rel_err(res[0][1], res[1][1]) <= GRAD_TOL
    for a, b in zip(res[0][2], res[1][2]):
        assert rel_err(a, b) <= GRAD_TOL


def test_split_backward_dense_and_chain_core_gradients_agree():
    """cfg5-class chain (H = 1024, d4 r8: split backward).  The hh core gradients accumulated densely
    (dW_hh^T = H_prev^T delta, then projected onto the cores) must equal the second-chain-pass route."""
    dev = torch.device("cuda:0")
    lib = _lib.load()
    torch.manual_seed(47)
    m = quiet(tr.TTLSTM, 256, 1024, 1, torch.device("cpu"), n_cores=4, tt_rank=8).to(dev)
    x = torch.rand(70, 9, 256, device=dev)
    h0 = 0.2 * torch.randn(70, 1024, device=dev)
    c0 = 0.2 * torch.randn(70, 1024, device=dev)
    w = torch.randn(70, 9, 1024, device=dev)
    res = []
    for flag, chunk in ((1, 4), (0, 0)):
        lib.ttrnn_set_option(b"dense_hh_dw", flag)
        lib.ttrnn_set_option(b"chunk_steps", chunk)
        try:
            for p in m.parameters():
                p.grad = None
            out, (h, c) = m(x, (h0, c0))
            ((out * w).sum() + c.sum()).backward()
            res.append([p.grad.clone() for p in m.parameters()])
        finally:
            lib.ttrnn_set_option(b"dense_hh_dw", 1)
            lib.ttrnn_set_option(b"chunk_steps", 0)
    for a, b in zip(res[0], res[1]):
        assert rel_err(a, b) <= GRAD_TOL


def test_split_kept_gates_backward_matches_fused():
    """d3r8 LSTM chain with kept gates: the dX-only recurrent kernel + dense accumulation of the hh core gradients
    (`split_kept`, default) against the fused BPTT kernel that accumulates the core gradients in registers."""
    dev = torch.device("cuda:0")
    lib = _lib.load()
    torch.manual_seed(53)
    m = quiet(tr.TTLSTM, 40, 256, 2, torch.device("cpu"), n_cores=3, tt_rank=8).to(dev)
    x = torch.rand(37, 11, 40, device=dev, requires_grad=True)
    h0 = 0.2 * torch.randn(37, 256, device=dev)
    c0 = 0.2 * torch.randn(37, 256, device=dev)
    w = torch.randn(37, 11, 256, device=dev)
    res = []
    for flag, chunk in ((1, 4), (0, 0)):
        lib.ttrnn_set_option(b"split_kept", flag)
        lib.ttrnn_set_option(b"chunk_steps", chunk)
        try:
            for p in m.parameters():
                p.grad = None
            x.grad = None
            h0r, c0r = h0.clone().requires_grad_(True), c0.clone().requires_grad_(True)
            out, (h, c) = m(x, (h0r, c0r))
            ((out * w).sum() + 2 * h.sum() + c.sum()).backward()
            res.append([x.grad.clone(), h0r.grad.clone(), c0r.grad.clone()] + [p.grad.clone() for p in m.parameters()])
        finally:
            lib.ttrnn_set_option(b"split_kept", 1)
            lib.ttrnn_set_option(b"chunk_steps", 0)
    for a, b in zip(res[0], res[1]):
        assert rel_err(a, b) <= GRAD_TOL


def test_two_phase_row_plan_matches_single_variant():
    """A batch that does not fill whole waves of the best BPTT variant runs in two phases (tail rows on a variant
    with fewer rows per CTA, row-offset pointers, shared gradient slots).  Must equal the one-variant launch."""
    dev = torch.device("cuda:0")
    lib = _lib.load()
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    B = 3 * sms + 2 * (sms // 2) + 1            # one full wave of 3-row CTAs plus a tail
    torch.manual_seed(43)
    m = quiet(tr.TTLSTM, 40, 256, 1, torch.device("cpu"), n_cores=3, tt_rank=8).to(dev)
    x = torch.rand(B, 5, 40, device=dev)
    h0 = 0.2 * torch.randn(B, 256, device=dev)
    c0 = 0.2 * torch.randn(B, 256, device=dev)
    w = torch.randn(B, 5, 256, device=dev)
    res = []
    for plan in (1, 0):
        lib.ttrnn_set_option(b"row_plan", plan)
        try:
            for p in m.parameters():
                p.grad = None
            h0r, c0r = h0.clone().requires_grad_(True), c0.clone().requires_grad_(True)
            out, (h, c) = m(x, (h0r, c0r))
            ((out * w).sum() + 2 * h.sum() + c.sum()).backward()
            res.append((out.detach().clone(), h0r.grad.clone(), c0r.grad.clone(), [p.grad.clone() for p in m.parameters()]))
        finally:
            lib.ttrnn_set_option(b"row_plan", 1)
    assert torch.equal(res[0][0], res[1][0])
    assert rel_err(res[0][1], res[1][1]) <= GRAD_TOL and rel_err(res[0][2], res[1][2]) <= GRAD_TOL
    for a, b in zip(res[0][3], res[1][3]):
        assert rel_err(a, b) <= GRAD_TOL


def test_static_and_runtime_shape_kernels_agree():
    """Same inputs through the static kernels and through the runtime-shape kernels (static_kernels=0)."""
    dev = torch.device("cuda:0")
    lib = _lib.load()
    torch.manual_seed(5)
    m = quiet(tr.TTGRU, 1, 256, 1, torch.device("cpu"), n_cores=2, tt_rank=4).to(dev)
    x = torch.rand(20, 30, 1, device=dev)
    res = []
    for flag in (1, 0):
        lib.ttrnn_set_option(b"static_kernels", flag)
        try:
            for p in m.parameters():
                p.grad = None
            out, h = m(x)
            (out.sum() + h.sum()).backward()
            res.append((out.detach().clone(), [p.grad.clone() for p in m.parameters()]))
        finally:
            lib.ttrnn_set_option(b"static_kernels", 1)
    assert rel_err(res[0][0], res[1][0]) <= FWD_TOL
    for a, b in zip(res[0][1], res[1][1]):
        assert rel_err(a, b) <= GRAD_TOL


def test_inference_mode_matches_training_forward():
    dev = torch.device("cuda:0")
    torch.manual_seed(6)
    m = quiet(tr.TTLSTM, 40, 256, 3, torch.device("cpu"), n_cores=3, tt_rank=8).to(dev)
    x = torch.rand(11, 7, 40, device=dev)
    out_a, (h_a, c_a) = m(x)
    with torch.no_grad():
        out_b, (h_b, c_b) = m(x)
    assert torch.equal(out_a.detach(), out_b) and torch.equal(h_a.detach(), h_b) and torch.equal(c_a.detach(), c_b)


def test_batch_sharding_reproduces_unsharded_gradients():
    """Fake world on one device: shard the batch 4 ways, sum the shard gradients, compare with the
    unsharded run (this is what the NCCL all-reduce of tensorized_rnn_b200.dist computes)."""
    from tensorized_rnn_b200.dist import shard_bounds
    dev = torch.device("cuda:0")
    torch.manual_seed(9)
    m = quiet(tr.TTLSTM, 40, 256, 3, torch.device("cpu"), n_cores=3, tt_rank=8).to(dev)
    params = list(m.parameters())
    x = torch.rand(22, 6, 40, device=dev)
    out, (h, c) = m(x)
    (h.sum() + 0.1 * out.sum()).backward()
    full = [p.grad.clone() for p in params]
    acc = [torch.zeros_like(p) for p in params]
    outs = []
    for r in range(4):
        lo, hi = shard_bounds(22, 4, r)
        for p in params:
            p.grad = None
        o, (hh, cc) = m(x[lo:hi])
        (hh.sum() + 0.1 * o.sum()).backward()
        outs.append(o.detach())
        for a, p in zip(acc, params):
            a += p.grad
    assert rel_err(torch.cat(outs), out) <= FWD_TOL
    for a, f in zip(acc, full):
        assert rel_err(a, f) <= GRAD_TOL
