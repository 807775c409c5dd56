"""Utterance-level embeddings without a GPU: the window table of `partial_windows` against a plain restatement of the
reference's rule (tests/utter_ref.py), the P = 160 table written out, argument validation, and the C-ABI surface
(ttrnn_partials_gather, ttrnn_segment_mean_normalize_forward / _backward)."""
import io
import os
import re
from contextlib import redirect_stdout

import numpy as np
import pytest
import torch

import tensorized_rnn_b200 as tr
from tensorized_rnn_b200 import _lib
from helpers import ROOT
from utter_ref import window_starts

SETTINGS = [(160, 0.5, 0.75), (165, 0.5, 0.75), (167, 0.5, 0.75), (160, 0.0, 1.0), (160, 0.9, 0.3), (1, 0.5, 0.75),
            (7, 0.25, 0.5), (40, 0.75, 0.01), (165, 0.5, 1.0)]


@pytest.mark.parametrize("P,overlap,min_coverage", SETTINGS)
def test_partial_windows_match_the_rule(P, overlap, min_coverage):
    lengths = list(range(1, 1201))
    first, valid, k = tr.partial_windows(lengths, P, overlap, min_coverage)
    assert first.dtype == np.int64 and valid.dtype == np.int32 and k.dtype == np.int64
    assert k.shape == (1200,) and first.shape == valid.shape == (int(k.sum()),)
    w, base = 0, 0
    for n, kn in zip(lengths, k):
        starts = window_starts(n, P, overlap, min_coverage)
        assert kn == len(starts), (n, kn, starts)
        assert first[w:w + kn].tolist() == [base + s for s in starts]
        assert valid[w:w + kn].tolist() == [min(P, n - s) for s in starts]
        w += kn
        base += n


def test_half_even_step():
    # 165 * 0.5 = 82.5 rounds to 82 and 167 * 0.5 = 83.5 to 84 (np.round, half to even)
    assert tr.partial_windows([400], 165)[0].tolist() == [0, 82, 164, 246]
    assert tr.partial_windows([400], 167)[0].tolist() == [0, 84, 168, 252]


def test_p160_table():
    table = {1: [0], 80: [0], 160: [0], 200: [0, 80], 240: [0, 80], 280: [0, 80, 160], 400: [0, 80, 160, 240],
             1000: [0, 80, 160, 240, 320, 400, 480, 560, 640, 720, 800, 880]}
    for n, starts in table.items():
        first, valid, k = tr.partial_windows([n])
        assert first.tolist() == starts and k.tolist() == [len(starts)]
        assert valid.tolist() == [min(160, n - s) for s in starts]
    # packed: the second utterance's windows start at its own first row
    first, valid, k = tr.partial_windows([200, 280])
    assert first.tolist() == [0, 80, 200, 280, 360] and valid.tolist() == [160, 120, 160, 160, 120] and k.tolist() == [2, 3]


@pytest.mark.parametrize("kw", [dict(partial_frames=0), dict(partial_frames=-3), dict(partial_frames=2.5),
                                dict(partial_frames=True), dict(overlap=1.0), dict(overlap=-0.1), dict(overlap=float("nan")),
                                dict(min_coverage=0.0), dict(min_coverage=1.5), dict(min_coverage=float("nan"))])
def test_partial_windows_rejects_bad_settings(kw):
    with pytest.raises(ValueError):
        tr.partial_windows([100, 200], **kw)


@pytest.mark.parametrize("lengths", [[], [0], [100, 0], [100, -5], [1.5], [[100]], [True]])
def test_partial_windows_rejects_bad_lengths(lengths):
    with pytest.raises(ValueError):
        tr.partial_windows(lengths)


def _encoder():
    torch.manual_seed(0)
    with redirect_stdout(io.StringIO()):
        return tr.SpeakerEncoder(40, 64, 1, 32, torch.device("cpu"), None, compression="tt", n_cores=3, rank=4)


def test_embed_utterances_validates_before_the_device():
    enc = _encoder()
    frames = torch.rand(300, 40)
    for lengths in ([100, 0, 200], [0], [], [100, 199], [100, 201]):
        with pytest.raises(ValueError):
            enc.embed_utterances(frames, lengths)
    with pytest.raises(ValueError):
        enc.embed_utterances(frames.view(1, 300, 40), [300])
    with pytest.raises(ValueError):
        enc.embed_utterances(frames, [300], overlap=1.0)
    with pytest.raises(RuntimeError):                  # valid arguments: the CPU tensor is refused, no fallback
        enc.embed_utterances(frames, [100, 200])
    with pytest.raises(NotImplementedError):           # the gather has no backward
        enc.embed_utterances(frames.requires_grad_(True), [100, 200])


def test_segment_and_gather_validation():
    x = torch.rand(6, 8)
    for counts in ([], [0, 6], [2, 3], [7], [2.0, 4.0]):
        with pytest.raises(ValueError):
            tr.segment_mean_normalize(x, counts)
    with pytest.raises(RuntimeError):
        tr.segment_mean_normalize(x, [2, 4])
    with pytest.raises(ValueError):
        _encoder().embed_speakers(x, [2, 3])
    frames = torch.rand(10, 4)
    for first, valid in (([0], [0]), ([0], [6]), ([8], [3]), ([-1], [2]), ([0, 1], [2]), ([], [])):
        with pytest.raises(ValueError):
            tr.gather_partials(frames, np.array(first, dtype=np.int64), np.array(valid, dtype=np.int32), 5)
    with pytest.raises(RuntimeError):
        tr.gather_partials(frames, np.array([0]), np.array([5]), 5)


def test_utterance_symbols_are_exported_and_declared():
    header = open(os.path.join(ROOT, "include", "ttrnn_b200.h")).read()
    lib = _lib.load()
    for name, nargs in (("ttrnn_partials_gather", 9), ("ttrnn_segment_mean_normalize_forward", 7),
                        ("ttrnn_segment_mean_normalize_backward", 8)):
        assert re.search(r"\bint %s\s*\(" % name, header), name
        assert len(_lib.SYMBOLS[name][1]) == nargs
        assert getattr(lib, name) is not None
    for name in ("partial_windows", "gather_partials", "segment_mean_normalize"):
        assert name in tr.__all__ and callable(getattr(tr, name))
    assert lib.ttrnn_abi_version() == _lib.ABI_VERSION == 4
