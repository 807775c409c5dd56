"""Row groups (round 2, second half): a multi-layer stack whose batch does not fill whole waves of CTAs is cut into
two independent row groups that run the stack on two streams (csrc/ttrnn_capi.cu, plan_row_groups).  The reference has
no counterpart (its layer loop, lstm.py:123-133, walks the whole batch), so the bar is the usual one: outputs, final
states and every gradient against the oracle on the same inputs (1e-5 forward / 1e-4 gradients, norm-wise relative),
for the planned split of the cfg3 shape and for forced splits of the other kernel families (GRU, rank-one input,
runtime-shape kernels, time chunks, non-zero initial states, gradient wrt the input and the initial states).
"""
import ctypes

import pytest
import torch

from tensorized_rnn_b200 import _lib
from helpers import FWD_TOL, GRAD_TOL, rel_err
from test_gpu_round2 import DEV, assert_grads, gpu_run, make_pair, options, oracle_run

pytestmark = pytest.mark.gpu


def planned_groups(m, B, T):
    rows = (ctypes.c_int64 * 2)()
    n = _lib.load().ttrnn_rnn_row_groups(ctypes.byref(m.spec().desc(B, T)), 0, rows)
    assert n >= 1, _lib.last_error()
    return n, rows[0], rows[1]


def test_planned_split_of_the_cfg3_shape_matches_oracle_and_single_group():
    """640 rows of the cfg3 stack on 148 SMs: the plan is 444 + 196 rows (one full wave of three-row CTAs, the rest at
    two rows per CTA).  T is short so that the oracle finishes in seconds; the split does not depend on T."""
    cell, I, H, L, d, r, B, T = "lstm", 40, 256, 3, 3, 8, 640, 6
    layers, m = make_pair(cell, I, H, L, d, r)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n, r0, r1 = planned_groups(m, B, T)
    if sms == 148:
        assert (n, r0, r1) == (2, 444, 196)
    g = torch.Generator().manual_seed(3)
    x = torch.rand(B, T, I, generator=g)
    w_out, w_h = torch.randn(B, T, H, generator=g), torch.randn(B, H, generator=g)
    o_ref, h_ref, g_ref = oracle_run(cell, layers, x, w_out, w_h)
    out, h, grads = gpu_run(cell, m, x, w_out, w_h)
    assert rel_err(out, o_ref) <= FWD_TOL and rel_err(h, h_ref) <= FWD_TOL
    assert_grads(grads, g_ref)
    with options(row_groups=0):
        assert planned_groups(m, B, T)[0] == 1
        out1, h1, grads1 = gpu_run(cell, m, x, w_out, w_h)
    # the two runs use different rows-per-CTA variants (summation order), so close, not bit-identical
    assert rel_err(out, out1) <= FWD_TOL and rel_err(h, h1) <= FWD_TOL
    assert_grads(grads, grads1)


FORCED = [
    # name, cell, I, H, L, d, r, B, T, rows of group 0, extra options
    ("gru_static_rank_one_input", "gru", 1, 256, 1, 2, 4, 40, 30, 24, {}),
    ("lstm_static_two_layers_rank_one_input", "lstm", 1, 256, 2, 2, 4, 36, 20, 20, {}),
    ("lstm_runtime_shape_kernels", "lstm", 12, 60, 2, 3, 3, 22, 9, 12, {}),
    ("gru_runtime_shape_kernels", "gru", 10, 48, 2, 2, 5, 17, 11, 8, {}),
    ("cfg3_shape_time_chunks", "lstm", 40, 256, 2, 3, 8, 44, 25, 28, {"chunk_steps": 10}),
    ("cfg3_shape_ffma_gemms", "lstm", 40, 256, 3, 3, 8, 40, 12, 16, {"tc_gemm": 0}),
    ("rank_padded_d2r2", "lstm", 40, 256, 2, 2, 2, 48, 10, 32, {}),
]


@pytest.mark.parametrize("case", FORCED, ids=[c[0] for c in FORCED])
def test_forced_split_matches_oracle(case):
    name, cell, I, H, L, d, r, B, T, rows0, extra = case
    layers, m = make_pair(cell, I, H, L, d, r)
    g = torch.Generator().manual_seed(11)
    x = torch.rand(B, T, I, generator=g)
    w_out, w_h = torch.randn(B, T, H, generator=g), torch.randn(B, H, generator=g)
    o_ref, h_ref, g_ref = oracle_run(cell, layers, x, w_out, w_h)
    with options(row_groups=rows0, **extra):
        n, r0, r1 = planned_groups(m, B, T)
        assert (n, r0, r1) == (2, rows0, B - rows0)
        out, h, grads = gpu_run(cell, m, x, w_out, w_h)
    assert rel_err(out, o_ref) <= FWD_TOL and rel_err(h, h_ref) <= FWD_TOL, (rel_err(out, o_ref), rel_err(h, h_ref))
    assert_grads(grads, g_ref)


@pytest.mark.parametrize("cell", ["lstm", "gru"])
def test_forced_split_with_initial_states_and_input_gradients(cell):
    """Every row-indexed pointer of the C ABI is sliced per group: h0 / c0, d_x, d_h0 / d_c0, h_T / c_T and their
    upstream gradients."""
    from helpers import oracle
    I, H, L, d, r, B, T, rows0 = 40, 256, 2, 3, 8, 28, 9, 16
    if cell == "gru":
        I, H, d, r = 16, 256, 2, 4
    layers, m = make_pair(cell, I, H, L, d, r)
    g = torch.Generator().manual_seed(21)
    x = torch.rand(B, T, I, generator=g)
    h0 = 0.5 * torch.randn(B, H, generator=g)
    c0 = 0.5 * torch.randn(B, H, generator=g)
    w_out, w_h, w_c = torch.randn(B, T, H, generator=g), torch.randn(B, H, generator=g), torch.randn(B, H, generator=g)

    def run(fwd, xs, hs, cs, dev):
        xs, hs, cs = (t.clone().to(dev).requires_grad_(True) for t in (xs, hs, cs))
        if cell == "lstm":
            out, (h, c) = fwd(xs, (hs, cs))
            loss = (out * w_out.to(dev)).sum() + (h * w_h.to(dev)).sum() + (c * w_c.to(dev)).sum()
        else:
            out, h = fwd(xs, hs)
            loss = (out * w_out.to(dev)).sum() + (h * w_h.to(dev)).sum()
        loss.backward()
        res = [out.detach(), h.detach(), xs.grad, hs.grad]
        if cell == "lstm":
            res.append(cs.grad)
        return res

    for p in oracle.flat_params(layers):
        p.grad = None
    fwd_ref = (lambda xs, st: oracle.lstm_forward(layers, xs, st)) if cell == "lstm" else (lambda xs, st: oracle.gru_forward(layers, xs, st))
    ref = run(fwd_ref, x, h0, c0, "cpu")
    g_ref = [p.grad.clone() for p in oracle.flat_params(layers)]
    for p in m.parameters():
        p.grad = None
    with options(row_groups=rows0):
        got = run(lambda xs, st: m(xs, st), x, h0, c0, DEV)
        torch.cuda.synchronize()
    assert rel_err(got[0], ref[0]) <= FWD_TOL and rel_err(got[1], ref[1]) <= FWD_TOL
    for a, b in zip(got[2:], ref[2:]):
        assert rel_err(a, b) <= GRAD_TOL, rel_err(a, b)
    assert_grads([p.grad for p in m.flat_parameters()], g_ref)


def test_split_inference_matches_training_forward():
    cell, I, H, L, d, r, B, T = "lstm", 40, 256, 3, 3, 8, 52, 14
    layers, m = make_pair(cell, I, H, L, d, r)
    x = torch.rand(B, T, I, generator=torch.Generator().manual_seed(2)).to(DEV)
    with options(row_groups=32):
        out_t, (h_t, c_t) = m(x)
        with torch.no_grad():
            out_i, (h_i, c_i) = m(x)
        torch.cuda.synchronize()
    with options(row_groups=0):
        with torch.no_grad():
            out_1, (h_1, c_1) = m(x)
        torch.cuda.synchronize()
    assert torch.equal(out_t, out_i) and torch.equal(h_t, h_i) and torch.equal(c_t, c_i)
    assert rel_err(out_i, out_1) <= FWD_TOL and rel_err(c_i, c_1) <= FWD_TOL


def test_options_changed_between_forward_and_backward_do_not_move_the_split():
    """The split is part of the plan stamped into the workspace struct: backward slices `saved` the way forward wrote it."""
    cell, I, H, L, d, r, B, T = "lstm", 40, 256, 2, 3, 8, 40, 10
    layers, m = make_pair(cell, I, H, L, d, r)
    g = torch.Generator().manual_seed(8)
    x = torch.rand(B, T, I, generator=g)
    w_h = torch.randn(B, H, generator=g)
    _, h_ref, g_ref = oracle_run(cell, layers, x, None, w_h)
    for p in m.parameters():
        p.grad = None
    lib = _lib.load()
    with options(row_groups=24):
        out, (h, _) = m(x.to(DEV))
        lib.ttrnn_set_option(b"row_groups", 0)                  # another model / thread changes the option here
        (h * w_h.to(DEV)).sum().backward()
        torch.cuda.synchronize()
    assert rel_err(h, h_ref) <= FWD_TOL
    assert_grads([p.grad for p in m.flat_parameters()], g_ref)


def recorded_recurrent_launches(m, x):
    """(kind, rows per CTA, CTAs, rows) of every recurrent-kernel launch of one forward + backward step, in issue order
    (kernel timing runs the row groups back to back on one stream)."""
    lib = _lib.load()
    kms, kcnt = (ctypes.c_double * 7)(), (ctypes.c_int64 * 7)()
    lib.ttrnn_kernel_times(kms, kcnt)
    lib.ttrnn_kernel_timing(1)
    try:
        m(x)[0].sum().backward()
        torch.cuda.synchronize()
    finally:
        lib.ttrnn_kernel_timing(0)
    lib.ttrnn_kernel_times(kms, kcnt)
    n = lib.ttrnn_kernel_launch_records(None, 0)
    buf = (ctypes.c_double * (6 * max(n, 1)))()
    lib.ttrnn_kernel_launch_records(buf, n)
    recs = [tuple(int(buf[6 * i + j]) for j in range(4)) for i in range(n)]
    return [r for r in recs if r[0] in (1, 2)]


def described_launches(plan, rows):
    """(kind, rows per CTA, rows) of the forward and backward recurrent launches that a describe_plan() result of a call
    on `rows` rows names."""
    fwd = [(1, lay["fwd_rows"], rows) for lay in plan[1:]]
    bwd = []
    for lay in reversed(plan[1:]):
        bwd.append((2, lay["bwd_rows"], lay["bwd_phase_rows"]))
        if "bwd_rows2" in lay:
            bwd.append((2, lay["bwd_rows2"], lay["bwd_phase_rows2"]))
    return fwd, bwd


DESCRIBED = [
    # name, cell, I, H, L, d, r, B, T, options
    ("cfg3_shape_640_rows", "lstm", 40, 256, 3, 3, 8, 640, 6, {}),
    ("cfg3_shape_640_rows_one_group", "lstm", 40, 256, 3, 3, 8, 640, 6, {"row_groups": 0}),
    ("cfg1_shape_256_rows", "lstm", 1, 256, 1, 2, 4, 256, 12, {}),
]


@pytest.mark.parametrize("case", DESCRIBED, ids=[c[0] for c in DESCRIBED])
def test_describe_matches_the_recorded_launches(case):
    """describe_plan() is what the tests and the benchmark read the kernel routes from: the recurrent launches of one
    training step must be the ones it names, per row group (rows per CTA, rows per launch, two-phase backward row plans,
    the CTAs of group 1), in issue order."""
    name, cell, I, H, L, d, r, B, T, extra = case
    _, m = make_pair(cell, I, H, L, d, r)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    x = torch.rand(B, T, I, generator=torch.Generator().manual_seed(5)).to(DEV)
    with options(**extra):
        plan = _lib.describe_plan(m.spec().desc(B, T), training=True)
        head = plan[0]
        groups = [head["group_rows0"], head["group_rows1"]] if head["row_groups"] == 2 else [B]
        plans = [plan]
        if len(groups) == 2:
            with options(row_groups=0):                    # group 1 runs the single-group routes of its own rows
                plans.append(_lib.describe_plan(m.spec().desc(groups[1], T), training=True))
        recs = recorded_recurrent_launches(m, x)
    if name == "cfg3_shape_640_rows" and sms == 148:
        assert groups == [444, 196], head
    if name == "cfg1_shape_256_rows":
        assert plan[1]["ih_route"] == "rank_one" and "split" in plan[1]["bwd_kernel"], plan[1]
    fwd, bwd = [], []
    for rows, p in zip(groups, plans):
        f, b = described_launches(p, rows)
        fwd += f
        bwd += b
    assert [rc[:2] + rc[3:] for rc in recs] == fwd + bwd, (plans, recs)
    for kind, R, ctas, rows in recs:
        tiles = -(-rows // R)
        assert ctas == tiles if tiles <= sms else sms <= ctas <= tiles, (kind, R, ctas, rows)
    if len(groups) == 2:
        g1_fwd, g1_bwd = recs[2 * L - 1], recs[2 * L + len(described_launches(plans[0], groups[0])[1])]
        assert (g1_fwd[2], g1_bwd[2]) == (head["group1_fwd_ctas"], head["group1_bwd_ctas"]), (head, recs)
