"""Plain restatements the utterance-embedding tests compare against: the window rule of `compute_partial_slices`
(Real-Time-Voice-Cloning, encoder/inference.py) counted in frames, one utterance at a time with Python loops, and the
FP64 composition of `SpeakerEncoder.embed_utterances` from `forward` on host-sliced windows."""
import numpy as np
import torch


def window_starts(n, P=160, overlap=0.5, min_coverage=0.75):
    """Window starts of one utterance of n frames, as the reference's loop computes them."""
    step = max(int(np.round(P * (1 - overlap))), 1)
    starts = list(range(0, max(1, n - P + step + 1), step))
    if len(starts) > 1 and (n - starts[-1]) / P < min_coverage:
        starts.pop()
    return starts


def windows_of(utt, P=160, overlap=0.5, min_coverage=0.75):
    """(k, P, F) windows of one (n, F) utterance, zero past its end (the reference pads the wav with zeros)."""
    n, F = utt.shape
    out = []
    for s in window_starts(n, P, overlap, min_coverage):
        w = torch.zeros(P, F, dtype=utt.dtype, device=utt.device)
        w[:min(P, n - s)] = utt[s:s + P]
        out.append(w)
    return torch.stack(out)


def mean_normalize64(rows, counts):
    """FP64 L2-normalised means of consecutive groups of rows."""
    out, r = [], 0
    for c in counts:
        m = rows[r:r + c].double().mean(dim=0)
        out.append(m / m.norm())
        r += c
    return torch.stack(out)
