"""Tensor-core stage 0 of the contracted d3 r8 dX-only BPTT kernel (csrc/tt_static.cuh, tts::TcStage0): the product
dX_0 = W01 dY_0 of every step runs as tcgen05 3xTF32 MMAs with W01 held in tensor memory.  The forward is untouched, so
it stays bit-identical to the three-core chain (`merge_cores = 0`); the gradients must agree with that FFMA reference at
1e-5 norm-wise at full cfg3 size, over a long sequence, and on ragged / partly empty row tiles at every rows-per-CTA R.
"""
import pytest
import torch

from helpers import rel_err
from test_gpu_merged_chain import layer_plans, opts
from test_gpu_round2 import assert_grads, gpu_run, make_pair, oracle_run

pytestmark = pytest.mark.gpu

I, H, d, r = 40, 256, 3, 8
TC_VS_3CORE_GRAD = 1e-5


def run_default_and_reference(m, x, w_out, w_h, **kw):
    res = {}
    for mc in (1, 0):
        with opts(merge_cores=mc, **kw):
            for lay in layer_plans(m, x.shape[0], x.shape[1]):
                assert ("(m01," in lay["bwd_kernel"]) == (mc == 1) and "split" in lay["bwd_kernel"], lay
            res[mc] = gpu_run("lstm", m, x, w_out, w_h)
    return res[1], res[0]


def check_against_reference(tc, ref3):
    out, h, grads = tc
    out0, h0, grads0 = ref3
    assert torch.equal(out, out0) and torch.equal(h, h0)
    assert_grads(grads, grads0, TC_VS_3CORE_GRAD)


def inputs(B, T, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(B, T, I, generator=g), torch.randn(B, T, H, generator=g) / (B * T) ** 0.5,
            torch.randn(B, H, generator=g) / B ** 0.5)


def test_cfg3_full_size():
    _, m = make_pair("lstm", I, H, 3, d, r, seed=31)
    x, w_out, w_h = inputs(640, 160, 32)
    check_against_reference(*run_default_and_reference(m, x, w_out, w_h))


def test_long_sequence():
    _, m = make_pair("lstm", I, H, 1, d, r, seed=41)
    x, w_out, w_h = inputs(3, 784, 42)
    check_against_reference(*run_default_and_reference(m, x, w_out, w_h))


# every R of the tensor-core kernel, with a ragged last row tile (B = 3R + 1) and with fewer rows than one tile (B < R)
CASES = [(rb, B) for rb in (1, 2, 3, 4) for B in sorted({3 * rb + 1, max(rb - 1, 1)})]


@pytest.mark.parametrize("rb,B", CASES, ids=["R%d_B%d" % c for c in CASES])
def test_ragged_and_partial_row_tiles(rb, B):
    L, T = 2, 6
    layers, m = make_pair("lstm", I, H, L, d, r, seed=50 + rb)
    x, w_out, w_h = inputs(B, T, 60 + B)
    with opts(static_rows_bwd=rb):
        for lay in layer_plans(m, B, T):
            assert lay["bwd_rows"] == rb, lay
    tc, ref3 = run_default_and_reference(m, x, w_out, w_h, static_rows_bwd=rb)
    check_against_reference(tc, ref3)
    o_ref, h_ref, g_ref = oracle_run("lstm", layers, x, w_out, w_h)
    assert rel_err(tc[0], o_ref) <= 1e-5 and rel_err(tc[1], h_ref) <= 1e-5
    assert_grads(tc[2], g_ref)
