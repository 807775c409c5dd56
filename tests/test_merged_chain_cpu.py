"""Contracted d3 r8 chain (tts::Merge01 in csrc/tt_static.cuh), host side.

The recurrent kernels of the d3 r8 TT-LSTM contract hh cores 0 and 1 while staging them and run the two-core chain
J = [32, 8], I = [64, 16], RK = [1, 8, 1].  The contraction below follows the kernel's index order (core_elem: blob
element e = (i, j, a2) of the merged core, i = i0 * I1 + i1, j = j0 * J1 + j1, sum over a1 in order); the dense W_hh of
the resulting two-core chain must be the oracle's dense W_hh of the three original cores.
"""
import ctypes

import numpy as np
import torch

from helpers import load_golden, oracle


def merge01_like_kernel(g0, g1):
    """(1, I0, J0, R1) x (R1, I1, J1, R2) -> (1, I0*I1, J0*J1, R2), element by element in the kernel's order."""
    _, I0, J0, R1 = g0.shape
    _, I1, J1, R2 = g1.shape
    out = np.zeros((1, I0 * I1, J0 * J1, R2), np.float32)
    for i in range(I0 * I1):
        for j in range(J0 * J1):
            for ap in range(R2):
                s = np.float32(0.0)
                for a1 in range(R1):
                    # fmaf(g0, g1, s): the product is exact in double, one rounding to float32 per step
                    s = np.float32(np.float64(g0[0, i // I1, j // J1, a1]) * np.float64(g1[a1, i % I1, j % J1, ap])
                                   + np.float64(s))
                out[0, i, j, ap] = s
    return out


def test_contracted_cores_give_the_oracle_dense_w_hh():
    g = load_golden("cfg3_lstm_d3r8_L3")
    for layer in range(3):
        cores = [g["param:cell%d.hidden_weights.parameters.%d" % (layer, k)].astype(np.float32) for k in range(3)]
        assert [c.shape for c in cores] == [(1, 8, 4, 8), (8, 8, 8, 8), (8, 16, 8, 1)]
        w01 = merge01_like_kernel(cores[0], cores[1])
        assert w01.shape == (1, 64, 32, 8)
        dense3 = oracle.tt_dense([torch.from_numpy(c).double() for c in cores]).numpy()
        dense2 = oracle.tt_dense([torch.from_numpy(w01).double(), torch.from_numpy(cores[2]).double()]).numpy()
        assert dense3.shape == dense2.shape == (1024, 256)
        assert np.linalg.norm(dense2 - dense3) / np.linalg.norm(dense3) <= 1e-6
        # and the two-core TT matvec of the oracle applies it the same way
        h = torch.from_numpy(np.random.default_rng(layer).standard_normal((5, 256))).double()
        y3 = oracle.tt_matvec([torch.from_numpy(c).double() for c in cores], h)
        y2 = oracle.tt_matvec([torch.from_numpy(w01).double(), torch.from_numpy(cores[2]).double()], h)
        assert float((y2 - y3).norm() / y3.norm()) <= 1e-6


def test_merge_cores_is_a_known_option():
    from tensorized_rnn_b200 import _lib
    lib = _lib.load()
    assert lib.ttrnn_set_option(b"merge_cores", 0) == 0
    assert lib.ttrnn_set_option(b"merge_cores", 1) == 0


def test_contracted_variants_are_registered_and_fit():
    """Forward R = 1..5 and dX-only backward R = 1..4 of the contracted chain, each under the 227 KB opt-in limit."""
    from tensorized_rnn_b200 import _lib
    lib = _lib.load()
    buf = ctypes.create_string_buffer(1 << 16)
    assert lib.ttrnn_static_kernel_table(buf, len(buf)) > 0
    rows = [ln.split("|") for ln in buf.value.decode().strip().splitlines()]
    m01 = [(k, int(R)) for k, name, R, smem, fits in rows if name.startswith("HH_H256_d3r8_lstm(m01") and fits == "1"]
    assert sorted(R for k, R in m01 if k == "rnn_fwd") == [1, 2, 3, 4, 5]
    assert sorted(R for k, R in m01 if k == "rnn_bwd") == [1, 2, 3, 4]
