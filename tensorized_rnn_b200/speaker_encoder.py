"""`SpeakerEncoder`: the GE2E speaker encoder of the reference with the recurrent stack, the projection and the GE2E head all
on the device.

Mirror of experiments/speaker_verification/encoder/speaker_encoder.py:17-170 -- same constructor signature, attribute and
sub-module names (`rnn`, `linear`, `similarity_weight`, `similarity_bias`: reference checkpoints load with `load_state_dict`),
`forward(utterances)` -> L2-normalised embeddings, `similarity_matrix`, `loss`, `do_gradient_ops`.  Differences: `loss_device` is
accepted and ignored (the reference moves the embeddings to the CPU for the loss, encoder/main.py:279-280; here the loss runs
in the CUDA library, ge2e.py); the EER, which the reference computes with scikit-learn on the CPU and does not backpropagate
(speaker_encoder.py:158-169), is computed the same way from a host copy of the similarity matrix only when `compute_eer=True`;
the evaluation form of `similarity_matrix` (`enrollment_embeds` given) is not provided by the CUDA head and raises.
`proj_size=P` (appended to the reference signature; LSTM only, the GRU modules refuse it) builds the LSTM with a recurrent
projection of the GE2E paper (LSTMP) on either side, `compression=None` (dense `LSTM`) or `'tt'` (`TTLSTM`); the embedding
`linear` then reads the P-wide final state.  `embed_utterances` / `embed_speakers` (appended) give the utterance and speaker
embeddings of enrollment and verification: sliding-window partials, embedded in one stack call and averaged (DESIGN.md §4.21),
or with `using_partials=False` each whole utterance embedded by one variable-length stack call (DESIGN.md §4.22).
"""
from __future__ import annotations

import numpy as np
import torch
from torch import nn

from .dense import GRU, LSTM
from .ge2e import _counts, embed_normalize, gather_partials, ge2e_loss, partial_windows, segment_mean_normalize
from .layers import TTLinear
from .rnn import TTGRU, TTLSTM


class SpeakerEncoder(nn.Module):
    def __init__(self, mel_n_channels, model_hidden_size, model_num_layers, model_embedding_size, device, loss_device=None,
                 compression=None, n_cores=3, rank=8, clip=3, use_gru=False, proj_size=0):
        super().__init__()
        state_size = proj_size or model_hidden_size
        self.loss_device = loss_device
        self.clip = clip
        self.use_gru = use_gru
        if compression is None:
            cls = GRU if use_gru else LSTM
            self.rnn = cls(mel_n_channels, model_hidden_size, model_num_layers, device, proj_size=proj_size)
            self.linear = nn.Linear(in_features=state_size, out_features=model_embedding_size).to(device)
        elif compression == 'tt':
            print("Encoding linear layer as a tensor-train...")
            if not use_gru:
                self.rnn = TTLSTM(mel_n_channels, model_hidden_size, model_num_layers, device, n_cores=n_cores, tt_rank=rank,
                                  proj_size=proj_size)
            else:
                self.rnn = TTGRU(mel_n_channels, model_hidden_size, model_num_layers, device, bias=True, n_cores=n_cores,
                                 tt_rank=rank, proj_size=proj_size)
            self.linear = TTLinear(in_features=state_size, out_features=model_embedding_size, bias=True,
                                   auto_shapes=True, d=n_cores, tt_rank=rank).to(device)
        else:
            raise ValueError("Unknown compression type: '{}'".format(compression))
        # cosine similarity scaling, fixed initial values (speaker_encoder.py:55-57)
        self.similarity_weight = nn.Parameter(torch.tensor([10.], device=device))
        self.similarity_bias = nn.Parameter(torch.tensor([-5.], device=device))

    def do_gradient_ops(self):
        self.similarity_weight.grad *= 0.01
        self.similarity_bias.grad *= 0.01
        torch.nn.utils.clip_grad_norm_(self.parameters(), self.clip, norm_type=2)

    def forward(self, utterances, hidden_init=None):
        return self._embed(self.rnn(utterances))

    def _embed(self, rnn_result):
        _, st = rnn_result
        last_hidden = st if self.use_gru else st[0]
        return embed_normalize(self.linear(last_hidden))            # relu + L2 norm (speaker_encoder.py:86-89)

    def embed_utterances(self, frames, lengths, partial_frames=160, overlap=0.5, min_coverage=0.75, using_partials=True):
        """Utterance d-vectors (N, E) of N utterances of any length, as GE2E and Real-Time-Voice-Cloning's `embed_utterance`
        define them: each utterance is cut into overlapping windows of `partial_frames` frames (`partial_windows`), every
        window is embedded by `forward`, and the window embeddings are averaged and L2-normalised.
        using_partials=False: the reference's full mode, `forward` on each whole utterance alone (ReLU + L2 norm of
        linear(h_n of the last layer)); the window arguments are then unused.

        frames: the utterances' frames packed in order, a CUDA float32 (sum(lengths), mel_n_channels) block (for a list of
        (n_i, mel) tensors: `torch.cat(utts)` with `[u.size(0) for u in utts]`); lengths: ints >= 1.  All windows of all
        utterances go through one gather, one `forward` and one segment mean (full mode: one window per utterance of
        max(lengths) frames, zero past the utterance, and one variable-length `forward`); the call is differentiable in
        the parameters."""
        n = _counts(lengths, "lengths")
        if frames.dim() != 2 or frames.shape[0] != int(n.sum()):
            raise ValueError("frames must be (sum(lengths) = %d, mel_n_channels), got %s" % (int(n.sum()), tuple(frames.shape)))
        if not using_partials:
            padded = gather_partials(frames, np.cumsum(n) - n, n.astype(np.int32), int(n.max()))
            return self._embed(self.rnn._forward_padded(padded, None, n))
        first, valid, n_windows = partial_windows(n, partial_frames, overlap, min_coverage)
        return segment_mean_normalize(self(gather_partials(frames, first, valid, partial_frames)), n_windows)

    def embed_speakers(self, d_vectors, counts):
        """Speaker embeddings (S, E): the L2-normalised mean of each group of `counts[s]` consecutive d-vector rows."""
        return segment_mean_normalize(d_vectors, counts)

    def similarity_matrix(self, verification_embeds, enrollment_embeds=None):
        if enrollment_embeds is not None:
            raise NotImplementedError("the device head implements the training form (enrollment = verification)")
        return ge2e_loss(verification_embeds, self.similarity_weight, self.similarity_bias, return_similarity=True)[1]

    def loss(self, verification_embeds, enrollment_embeds=None, compute_eer=False, group=None):
        """Returns (loss, eer): eer is None unless compute_eer (it needs a device-to-host copy and scikit-learn)."""
        if enrollment_embeds is not None:
            raise NotImplementedError("the device head implements the training form (enrollment = verification)")
        if not compute_eer:
            return ge2e_loss(verification_embeds, self.similarity_weight, self.similarity_bias, group=group), None
        loss, sim = ge2e_loss(verification_embeds, self.similarity_weight, self.similarity_bias, group=group,
                              return_similarity=True)
        from scipy.interpolate import interp1d
        from scipy.optimize import brentq
        from sklearn.metrics import roc_curve
        S, U = sim.shape[0], sim.shape[1]
        labels = np.eye(S, dtype=np.int64)[np.repeat(np.arange(S), U)]
        preds = sim.detach().reshape(S * U, S).cpu().numpy()
        fpr, tpr, _ = roc_curve(labels.flatten(), preds.flatten())
        eer = brentq(lambda x: 1. - x - interp1d(fpr, tpr)(x), 0., 1.)
        return loss, eer
