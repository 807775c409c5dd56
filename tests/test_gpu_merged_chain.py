"""Contracted d3 r8 chain (csrc/tt_static.cuh, tts::Merge01): the static kernels of the d3 r8 TT-LSTM contract cores 0
and 1 while staging them and run a two-core chain.  `merge_cores` = 1 (default): the dX-only BPTT kernels only, the forward
stays on the three-core chain and its results are bit-identical to `merge_cores = 0`; 2: the forward kernels as well.
Every case runs against the oracle (1e-5 forward / 1e-4 gradients, norm-wise relative) and against `merge_cores = 0` on
the same inputs: the routes differ only in the order of the sums and in one rounding per contracted weight, so they must
agree far inside the oracle bars.
"""
import contextlib

import pytest
import torch

from tensorized_rnn_b200 import _lib
from helpers import FWD_TOL, GRAD_TOL, oracle, rel_err
from test_gpu_round2 import DEV, assert_grads, gpu_run, make_pair, oracle_run

pytestmark = pytest.mark.gpu

I, H, d, r = 40, 256, 3, 8
MERGED_VS_3CORE = 1e-5         # forward, merged against the three-core chain (measured ~1e-7)
MERGED_VS_3CORE_GRAD = 1e-5    # gradients, same


@contextlib.contextmanager
def opts(**kw):
    defaults = {"merge_cores": 1, "static_rows_fwd": 0, "static_rows_bwd": 0, "row_groups": 1}
    lib = _lib.load()
    for k, v in kw.items():
        assert lib.ttrnn_set_option(k.encode(), int(v)) == 0, k
    try:
        yield lib
    finally:
        for k in kw:
            lib.ttrnn_set_option(k.encode(), defaults[k])


def layer_plans(m, B, T, training=True):
    return _lib.describe_plan(m.spec().desc(B, T), training=training)[1:]


def run_both(m, x, w_out, w_h, level=2, **kw):
    """(merged at `level`, three-core) results of the same training step under the options `kw`, kernels checked."""
    res = {}
    for mc in (level, 0):
        with opts(merge_cores=mc, **kw):
            B, T = x.shape[0], x.shape[1]
            for lay in layer_plans(m, B, T):
                assert ("(m01" in lay["fwd_kernel"]) == (mc >= 2), lay
                assert ("(m01" in lay["bwd_kernel"]) == (mc >= 1), lay
                assert "split" in lay["bwd_kernel"], lay
            res[mc] = gpu_run("lstm", m, x, w_out, w_h)
    return res[level], res[0]


def check(merged, plain, ref, level=2):
    out, h, grads = merged
    out0, h0, grads0 = plain
    o_ref, h_ref, g_ref = ref
    assert rel_err(out, o_ref) <= FWD_TOL and rel_err(h, h_ref) <= FWD_TOL, (rel_err(out, o_ref), rel_err(h, h_ref))
    assert_grads(grads, g_ref)
    if level == 1:      # forward on the three-core chain: bit-identical
        assert torch.equal(out, out0) and torch.equal(h, h0)
    assert rel_err(out, out0) <= MERGED_VS_3CORE and rel_err(h, h0) <= MERGED_VS_3CORE
    assert_grads(grads, grads0, MERGED_VS_3CORE_GRAD)


# forced rows-per-CTA variants: forward R = 1..5, dX-only backward R = 1..4 (R = 4 is registered for the merged chain
# only; the three-core run then takes its own pick).  B leaves a ragged last row tile for every R > 1.
ROWS = [(1, 1), (2, 2), (3, 3), (4, 4), (5, 3)]


@pytest.mark.parametrize("rf,rb", ROWS, ids=["fwd%d_bwd%d" % rr for rr in ROWS])
def test_every_registered_row_variant(rf, rb):
    L, T = 2, 7
    B = 2 * max(rf, rb) * 3 + 1
    layers, m = make_pair("lstm", I, H, L, d, r)
    g = torch.Generator().manual_seed(100 + rf)
    x = torch.rand(B, T, I, generator=g)
    w_out, w_h = torch.randn(B, T, H, generator=g), torch.randn(B, H, generator=g)
    ref = oracle_run("lstm", layers, x, w_out, w_h)
    with opts(merge_cores=2, static_rows_fwd=rf, static_rows_bwd=rb):
        lay = layer_plans(m, B, T)[0]
        assert lay["fwd_rows"] == rf and lay["bwd_rows"] == rb, lay
    merged, plain = run_both(m, x, w_out, w_h, 2, static_rows_fwd=rf, static_rows_bwd=rb)
    check(merged, plain, ref)


@pytest.mark.parametrize("level", [1, 2], ids=["bwd_only", "fwd_and_bwd"])
@pytest.mark.parametrize("B,T", [(13, 1), (29, 12)], ids=["T1", "T12"])
def test_planned_variants_short_sequences(B, T, level):
    layers, m = make_pair("lstm", I, H, 3, d, r, seed=7)
    g = torch.Generator().manual_seed(B)
    x = torch.rand(B, T, I, generator=g)
    w_out, w_h = torch.randn(B, T, H, generator=g), torch.randn(B, H, generator=g)
    ref = oracle_run("lstm", layers, x, w_out, w_h)
    check(*run_both(m, x, w_out, w_h, level), ref, level)


@pytest.mark.parametrize("level", [1, 2], ids=["bwd_only", "fwd_and_bwd"])
def test_forced_row_group_cut(level):
    L, B, T, rows0 = 3, 44, 9, 28
    layers, m = make_pair("lstm", I, H, L, d, r, seed=5)
    g = torch.Generator().manual_seed(17)
    x = torch.rand(B, T, I, generator=g)
    w_out, w_h = torch.randn(B, T, H, generator=g), torch.randn(B, H, generator=g)
    ref = oracle_run("lstm", layers, x, w_out, w_h)
    check(*run_both(m, x, w_out, w_h, level, row_groups=rows0), ref, level)


def test_default_keeps_the_forward_bit_identical():
    """merge_cores = 1 (the default) only reorders the BPTT sums: every forward result is the three-core chain's."""
    L, B, T = 3, 31, 10
    layers, m = make_pair("lstm", I, H, L, d, r, seed=21)
    g = torch.Generator().manual_seed(22)
    x = torch.rand(B, T, I, generator=g)
    w_out, w_h = torch.randn(B, T, H, generator=g), torch.randn(B, H, generator=g)
    ref = oracle_run("lstm", layers, x, w_out, w_h)
    with opts():
        lay = layer_plans(m, B, T)[0]
        assert "(m01" not in lay["fwd_kernel"] and "(m01" in lay["bwd_kernel"], lay
    check(*run_both(m, x, w_out, w_h, 1), ref, 1)


@pytest.mark.parametrize("with_init", [True, False], ids=["init_states", "zero_states"])
def test_initial_states_and_their_gradients(with_init):
    L, B, T = 2, 23, 8
    layers, m = make_pair("lstm", I, H, L, d, r, seed=9)
    g = torch.Generator().manual_seed(31)
    x = torch.rand(B, T, I, generator=g)
    h0 = 0.5 * torch.randn(B, H, generator=g)
    c0 = 0.5 * torch.randn(B, H, generator=g)
    w_out, w_h, w_c = torch.randn(B, T, H, generator=g), torch.randn(B, H, generator=g), torch.randn(B, H, generator=g)

    def run(fwd, params, dev):
        for p in params:
            p.grad = None
        xs = x.clone().to(dev).requires_grad_(True)
        hs = h0.clone().to(dev).requires_grad_(True)
        cs = c0.clone().to(dev).requires_grad_(True)
        out, (h, c) = fwd(xs, (hs, cs)) if with_init else fwd(xs, None)
        loss = (out * w_out.to(dev)).sum() + (h * w_h.to(dev)).sum() + (c * w_c.to(dev)).sum()
        loss.backward()
        res = [out.detach(), h.detach(), c.detach(), xs.grad]
        if with_init:
            res += [hs.grad, cs.grad]
        return res + [p.grad.clone() for p in params]

    ref = run(lambda xs, st: oracle.lstm_forward(layers, xs, st), oracle.flat_params(layers), "cpu")
    got = {}
    for mc in (2, 1, 0):
        with opts(merge_cores=mc):
            got[mc] = run(lambda xs, st: m(xs, st), list(m.flat_parameters()), DEV)
            torch.cuda.synchronize()
    for res in got.values():
        for i, (a, b) in enumerate(zip(res, ref)):
            assert rel_err(a, b) <= (FWD_TOL if i < 3 else GRAD_TOL), (i, rel_err(a, b))
    for mc in (2, 1):
        for i, (a, b) in enumerate(zip(got[mc], got[0])):
            assert rel_err(a, b) <= MERGED_VS_3CORE, (mc, i, rel_err(a, b))
            if mc == 1 and i < 3:
                assert torch.equal(a, b), (i, rel_err(a, b))


def test_inference_forward_matches_training_forward():
    L, B, T = 3, 37, 11
    layers, m = make_pair("lstm", I, H, L, d, r, seed=3)
    x = torch.rand(B, T, I, generator=torch.Generator().manual_seed(4)).to(DEV)
    with opts(merge_cores=2):
        for lay in layer_plans(m, B, T, training=False):
            assert "(m01)" in lay["fwd_kernel"], lay
        out_t, (h_t, c_t) = m(x)
        with torch.no_grad():
            out_i, (h_i, c_i) = m(x)
    with torch.no_grad():
        with opts(merge_cores=0):
            out_0, (h_0, c_0) = m(x)
        o_ref, (h_ref, c_ref) = oracle.lstm_forward(layers, x.cpu())
    torch.cuda.synchronize()
    # same kernel, same arithmetic: the kept-gates stores of the training forward are the only difference
    assert torch.equal(out_i, out_t.detach()) and torch.equal(h_i, h_t.detach()) and torch.equal(c_i, c_t.detach())
    assert rel_err(out_i, o_ref) <= FWD_TOL and rel_err(h_i, h_ref) <= FWD_TOL and rel_err(c_i, c_ref) <= FWD_TOL
    assert rel_err(out_i, out_0) <= MERGED_VS_3CORE and rel_err(c_i, c_0) <= MERGED_VS_3CORE


def test_backward_follows_the_plan_of_its_forward():
    """merge_cores is stamped into the workspace plan: switching it between a forward and its backward changes neither."""
    L, B, T = 2, 20, 6
    layers, m = make_pair("lstm", I, H, L, d, r, seed=12)
    g = torch.Generator().manual_seed(13)
    x = torch.rand(B, T, I, generator=g)
    w_h = torch.randn(B, H, generator=g)
    _, h_ref, g_ref = oracle_run("lstm", layers, x, None, w_h)
    for mc in (2, 0):
        for p in m.parameters():
            p.grad = None
        with opts(merge_cores=mc):
            out, (h, _) = m(x.to(DEV))
        with opts(merge_cores=2 - mc):
            (h * w_h.to(DEV)).sum().backward()
        torch.cuda.synchronize()
        assert rel_err(h, h_ref) <= FWD_TOL
        assert_grads([p.grad for p in m.flat_parameters()], g_ref)
