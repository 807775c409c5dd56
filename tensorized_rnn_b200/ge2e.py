"""GE2E head on the device (SURVEY.md 8f-4): embedding normalisation and the GE2E softmax loss.

Mirrors the training path of the reference's `SpeakerEncoder` (experiments/speaker_verification/encoder/
speaker_encoder.py): `forward` ends with ReLU + L2 normalisation (:86-89); `similarity_matrix` (:93-141) and `loss`
(:143-156) build inclusive / exclusive centroids, the scaled cosine-similarity matrix and the cross-entropy.  The
reference moves the embeddings to the CPU for this (encoder/main.py:279-280); here it stays on the GPU, in the CUDA
library (`ttrnn_embed_*`, `ttrnn_ge2e_loss_*`), with hand-written backward kernels.  Under data parallelism the loss
couples every speaker of the global batch: `ge2e_loss(..., group=...)` all-gathers the embeddings (NCCL), every
rank evaluates the full loss and keeps the gradient rows of its own utterances.

Utterance-level embeddings (DESIGN.md §4.21): `partial_windows` cuts utterances of any length into the fixed-length windows
the encoder trains on, `gather_partials` builds the window block on the device and `segment_mean_normalize` averages and
L2-normalises the window embeddings of each utterance (or the d-vectors of each speaker).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch
from torch import nn

from . import _lib
from .functional import _dense16, _ptr, _require_cuda_f32


class _EmbedNormalize(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        lib = _lib.load()
        _require_cuda_f32("embeddings", x)
        if x.dim() != 2:
            raise ValueError("embeddings must be (rows, features), got %s" % (tuple(x.shape),))
        x = _dense16(x)
        rows, E = x.shape
        with torch.cuda.device(x.device):
            y = torch.empty_like(x)
            inv = torch.empty(rows, device=x.device, dtype=torch.float32)
            stream = torch.cuda.current_stream(x.device).cuda_stream
            _lib.check(lib.ttrnn_embed_forward(rows, E, _ptr(x), _ptr(y), _ptr(inv), stream), "ttrnn_embed_forward")
        ctx.save_for_backward(x, y, inv)
        return y

    @staticmethod
    def backward(ctx, dy):
        lib = _lib.load()
        x, y, inv = ctx.saved_tensors
        dy = _dense16(dy)
        rows, E = x.shape
        with torch.cuda.device(x.device):
            dx = torch.empty_like(x)
            stream = torch.cuda.current_stream(x.device).cuda_stream
            _lib.check(lib.ttrnn_embed_backward(rows, E, _ptr(x), _ptr(y), _ptr(inv), _ptr(dy), _ptr(dx), stream),
                       "ttrnn_embed_backward")
        return dx


def embed_normalize(x: torch.Tensor) -> torch.Tensor:
    """relu(x) / ||relu(x)||_2 per row (speaker_encoder.py:86-89)."""
    return _EmbedNormalize.apply(x)


class _Ge2eLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, embeds, wb, want_sim: bool):
        lib = _lib.load()
        _require_cuda_f32("embeds", embeds)
        _require_cuda_f32("similarity weight / bias", wb)
        if embeds.dim() != 3:
            raise ValueError("embeds must be (speakers, utterances, features), got %s" % (tuple(embeds.shape),))
        S, U, E = embeds.shape
        embeds = _dense16(embeds)
        wb = _dense16(wb)
        with torch.cuda.device(embeds.device):
            nbytes = lib.ttrnn_ge2e_workspace_bytes(S, U, E)
            if nbytes < 0:
                raise ValueError("ttrnn_ge2e_workspace_bytes failed: " + _lib.last_error())
            ws = torch.empty((nbytes + 3) // 4, device=embeds.device, dtype=torch.float32)
            loss = torch.empty((), device=embeds.device, dtype=torch.float32)
            sim = torch.empty((S, U, S), device=embeds.device, dtype=torch.float32) if want_sim else None
            stream = torch.cuda.current_stream(embeds.device).cuda_stream
            _lib.check(lib.ttrnn_ge2e_loss_forward(S, U, E, _ptr(embeds), _ptr(wb), _ptr(loss), _ptr(sim), _ptr(ws), stream),
                       "ttrnn_ge2e_loss_forward")
        ctx.save_for_backward(embeds, wb, ws)
        if want_sim:
            ctx.mark_non_differentiable(sim)
            return loss, sim
        return loss, None

    @staticmethod
    def backward(ctx, dloss, _dsim):
        lib = _lib.load()
        embeds, wb, ws = ctx.saved_tensors
        S, U, E = embeds.shape
        with torch.cuda.device(embeds.device):
            g = _dense16(dloss.reshape(1).to(torch.float32))
            d_embeds = torch.empty_like(embeds)
            d_wb = torch.empty(2, device=embeds.device, dtype=torch.float32)
            stream = torch.cuda.current_stream(embeds.device).cuda_stream
            _lib.check(lib.ttrnn_ge2e_loss_backward(S, U, E, _ptr(embeds), _ptr(wb), _ptr(g), _ptr(ws), _ptr(d_embeds),
                                                    _ptr(d_wb), stream), "ttrnn_ge2e_loss_backward")
        return d_embeds, d_wb, None


class _AllGatherRows(torch.autograd.Function):
    """all_gather along dim 0 whose backward keeps this rank's rows of the (replicated) gradient."""

    @staticmethod
    def forward(ctx, x, group):
        import torch.distributed as dist
        world = dist.get_world_size(group)
        ctx.rank, ctx.n = dist.get_rank(group), x.shape[0]
        parts = [torch.empty_like(x) for _ in range(world)]
        dist.all_gather(parts, x.contiguous(), group=group)
        return torch.cat(parts, dim=0)

    @staticmethod
    def backward(ctx, g):
        return g[ctx.rank * ctx.n:(ctx.rank + 1) * ctx.n].contiguous(), None


def ge2e_loss(embeds: torch.Tensor, similarity_weight: torch.Tensor, similarity_bias: torch.Tensor,
              group=None, return_similarity: bool = False):
    """GE2E softmax loss of `embeds` (speakers, utterances, features), enrollment = verification (the training form).

    With `group` (a torch.distributed process group whose ranks each hold a contiguous block of speakers) the
    embeddings are all-gathered first; every rank then computes the loss of the GLOBAL batch, and autograd hands
    each rank the gradient rows of its own speakers.  Returns the loss (0-dim) [and the scaled similarity matrix]."""
    if group is not None:
        embeds = _AllGatherRows.apply(embeds, group)
    wb = torch.cat([similarity_weight.reshape(1), similarity_bias.reshape(1)])
    loss, sim = _Ge2eLoss.apply(embeds, wb, bool(return_similarity))
    return (loss, sim) if return_similarity else loss


def _counts(v, what: str) -> np.ndarray:
    """A 1-D host sequence of ints >= 1 (a list, a numpy array or a CPU tensor) as int64."""
    a = np.asarray(v.tolist() if isinstance(v, torch.Tensor) else v)
    if a.ndim != 1 or a.size == 0 or a.dtype.kind not in "iu":
        raise ValueError("%s must be a non-empty 1-D sequence of ints, got %r" % (what, v))
    if (a < 1).any():
        raise ValueError("every entry of %s must be >= 1, got %r" % (what, v))
    return a.astype(np.int64)


def partial_windows(lengths, partial_frames: int = 160, overlap: float = 0.5, min_coverage: float = 0.75):
    """Window table of `compute_partial_slices` (Real-Time-Voice-Cloning, encoder/inference.py), in frames.

    For an utterance of n >= 1 frames and P = partial_frames: step = max(round_half_even(P * (1 - overlap)), 1); the
    window starts are range(0, max(1, n - P + step + 1), step); when there is more than one window and
    (n - last_start) / P < min_coverage, the last window is dropped.  The utterances are packed in order, so window w
    covers packed rows first[w] .. first[w] + valid[w] - 1 and is zero past them (valid = min(P, n - start)).

    Host only.  Returns (first int64, valid int32, windows per utterance int64), numpy arrays."""
    if isinstance(partial_frames, bool) or not isinstance(partial_frames, (int, np.integer)) or partial_frames < 1:
        raise ValueError("partial_frames must be an int >= 1, got %r" % (partial_frames,))
    if not 0.0 <= overlap < 1.0:
        raise ValueError("overlap must be in [0, 1), got %r" % (overlap,))
    if not 0.0 < min_coverage <= 1.0:
        raise ValueError("min_coverage must be in (0, 1], got %r" % (min_coverage,))
    n = _counts(lengths, "lengths")
    P = int(partial_frames)
    step = max(int(np.round(P * (1 - overlap))), 1)
    k = (np.maximum(1, n - P + step + 1) + step - 1) // step
    k -= (k > 1) & ((n - (k - 1) * step) / P < min_coverage)
    utt = np.repeat(np.arange(n.size), k)
    start = (np.arange(int(k.sum())) - np.repeat(np.cumsum(k) - k, k)) * step
    first = (np.cumsum(n) - n)[utt] + start
    valid = np.minimum(P, n[utt] - start)
    assert (valid >= 1).all()
    return first.astype(np.int64), valid.astype(np.int32), k


def gather_partials(frames: torch.Tensor, first, valid, partial_frames: int) -> torch.Tensor:
    """(W, partial_frames, F) window block from the packed frames (total_frames, F) and a window table (`partial_windows`):
    window w holds rows first[w] .. first[w] + valid[w] - 1 and zeros after them.  A copy on the device
    (`ttrnn_partials_gather`), without autograd: the frames are model inputs."""
    if frames.requires_grad:
        raise NotImplementedError("gather_partials has no backward: the frames must not require grad")
    first, valid = np.asarray(first), np.asarray(valid)
    if first.ndim != 1 or first.size == 0 or first.shape != valid.shape or first.dtype.kind not in "iu" \
            or valid.dtype.kind not in "iu":
        raise ValueError("first / valid must be two non-empty 1-D int arrays of one length")
    if frames.dim() != 2:
        raise ValueError("frames must be (total_frames, features), got %s" % (tuple(frames.shape),))
    P = int(partial_frames)
    total, F = frames.shape
    if P < 1 or (valid < 1).any() or (valid > P).any() or (first < 0).any() or (first + valid > total).any():
        raise ValueError("window table out of range: need 1 <= valid <= partial_frames and first + valid <= %d" % total)
    lib = _lib.load()
    _require_cuda_f32("frames", frames)
    frames = _dense16(frames)
    W = first.size
    with torch.cuda.device(frames.device):
        out = torch.empty((W, P, F), device=frames.device, dtype=torch.float32)
        first_d = torch.from_numpy(first.astype(np.int64)).to(frames.device)
        valid_d = torch.from_numpy(valid.astype(np.int32)).to(frames.device)
        stream = torch.cuda.current_stream(frames.device).cuda_stream
        _lib.check(lib.ttrnn_partials_gather(W, P, F, _ptr(frames), total, _ptr(first_d), _ptr(valid_d), _ptr(out), stream),
                   "ttrnn_partials_gather")
    return out


class _SegmentMeanNormalize(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, off):
        lib = _lib.load()
        x = _dense16(x)
        n_seg, (rows, E) = off.numel() - 1, x.shape
        with torch.cuda.device(x.device):
            y = torch.empty((n_seg, E), device=x.device, dtype=torch.float32)
            inv = torch.empty(n_seg, device=x.device, dtype=torch.float32)
            stream = torch.cuda.current_stream(x.device).cuda_stream
            _lib.check(lib.ttrnn_segment_mean_normalize_forward(n_seg, E, _ptr(x), _ptr(off), _ptr(y), _ptr(inv), stream),
                       "ttrnn_segment_mean_normalize_forward")
        ctx.save_for_backward(off, y, inv)
        ctx.rows = rows
        return y

    @staticmethod
    def backward(ctx, dy):
        lib = _lib.load()
        off, y, inv = ctx.saved_tensors
        dy = _dense16(dy)
        n_seg, E = y.shape
        with torch.cuda.device(y.device):
            dx = torch.empty((ctx.rows, E), device=y.device, dtype=torch.float32)
            stream = torch.cuda.current_stream(y.device).cuda_stream
            _lib.check(lib.ttrnn_segment_mean_normalize_backward(n_seg, E, _ptr(off), _ptr(y), _ptr(inv), _ptr(dy), _ptr(dx),
                                                                 stream), "ttrnn_segment_mean_normalize_backward")
        return dx, None


def segment_mean_normalize(x: torch.Tensor, counts) -> torch.Tensor:
    """L2-normalised means of consecutive row groups: x (R, E), counts (S,) of ints >= 1 summing to R -> (S, E), row s the
    normalised mean of the counts[s] rows after the first sum(counts[:s]).  Differentiable (`ttrnn_segment_mean_normalize_*`)."""
    c = _counts(counts, "counts")
    if x.dim() != 2:
        raise ValueError("x must be (rows, features), got %s" % (tuple(x.shape),))
    if int(c.sum()) != x.shape[0]:
        raise ValueError("counts sum to %d, but x has %d rows" % (int(c.sum()), x.shape[0]))
    _require_cuda_f32("x", x)
    off = torch.from_numpy(np.concatenate([[0], np.cumsum(c)])).to(x.device)
    return _SegmentMeanNormalize.apply(x, off)


class GE2EHead(nn.Module):
    """ReLU + L2 normalisation and the GE2E loss with the reference's learnable similarity scale
    (speaker_encoder.py:52-57: weight 10, bias -5).  `forward(x)` -> embeddings; `loss(embeds)` -> loss."""

    def __init__(self, device=None):
        super().__init__()
        self.similarity_weight = nn.Parameter(torch.tensor([10.], device=device))
        self.similarity_bias = nn.Parameter(torch.tensor([-5.], device=device))

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return embed_normalize(x)

    def similarity_matrix(self, embeds: torch.Tensor) -> torch.Tensor:
        return ge2e_loss(embeds, self.similarity_weight, self.similarity_bias, return_similarity=True)[1]

    def loss(self, embeds: torch.Tensor, group=None) -> torch.Tensor:
        return ge2e_loss(embeds, self.similarity_weight, self.similarity_bias, group=group)

    def do_gradient_ops(self, parameters, clip: float = 3.0):
        """Gradient scale of the similarity parameters and global-norm clipping (speaker_encoder.py:62-68)."""
        self.similarity_weight.grad *= 0.01
        self.similarity_bias.grad *= 0.01
        torch.nn.utils.clip_grad_norm_(parameters, clip, norm_type=2)
