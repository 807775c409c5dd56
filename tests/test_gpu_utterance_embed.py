"""Utterance-level embeddings on the device: the window gather bit for bit against torch indexing, the segment mean +
normalisation and its backward against FP64, and `SpeakerEncoder.embed_utterances` / `embed_speakers` against the
composition of `forward` on host-sliced windows (tests/utter_ref.py) with the mean and normalisation in FP64, for the
reference weights of the three spkenc_* fixtures and for projected encoders."""
import glob
import io
import os
from contextlib import redirect_stdout

import numpy as np
import pytest
import torch

import tensorized_rnn_b200 as tr
from helpers import FWD_TOL, GOLDEN, GRAD_TOL, rel_err
from utter_ref import mean_normalize64, windows_of

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
CPU = torch.device("cpu")


def _sms():
    return torch.cuda.get_device_properties(DEV).multi_processor_count


def _lengths(seed, n, hi, fixed=()):
    g = np.random.default_rng(seed)
    return list(fixed) + g.integers(1, hi + 1, size=n).tolist()


def _gather_ref(frames, first, valid, P):
    W, F = first.size, frames.shape[1]
    ref = torch.zeros(W, P, F, device=frames.device)
    t = torch.arange(P, device=frames.device)
    first_d = torch.from_numpy(first).to(frames.device)
    mask = t[None, :] < torch.from_numpy(valid.astype(np.int64)).to(frames.device)[:, None]
    ref[mask] = frames[(first_d[:, None] + t[None, :])[mask]]
    return ref


# ---- gather --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("F", [40, 13])
@pytest.mark.parametrize("P,overlap,min_coverage", [(160, 0.5, 0.75), (7, 0.25, 0.5), (160, 0.0, 1.0)])
def test_gather_is_exact(F, P, overlap, min_coverage):
    lengths = _lengths(1, 400, 3000, fixed=(1, 5, P - 1, P, P + 1, 2 * P + 3))
    first, valid, k = tr.partial_windows(lengths, P, overlap, min_coverage)
    frames = torch.randn(sum(lengths), F, device=DEV)
    out = tr.gather_partials(frames, first, valid, P)
    assert out.shape == (first.size, P, F)
    assert torch.equal(out, _gather_ref(frames, first, valid, P))
    assert (valid < P).any() and (k == 1).any()          # windows past the end, utterances shorter than P
    if P == 160:
        assert first.size > 8 * _sms()                    # more windows than the grid (one CTA per window, 8 per SM)
    # a gather out of a slice of a larger block reads only the rows it is given
    big = torch.randn(sum(lengths) + 9, F, device=DEV)
    assert torch.equal(tr.gather_partials(big[4:4 + sum(lengths)], first, valid, P),
                       _gather_ref(big[4:4 + sum(lengths)], first, valid, P))


# ---- segment mean + normalisation ------------------------------------------------------------------------------------------
def _segment_cases():
    g = np.random.default_rng(2)
    mixed = [1] * 20 + [3000] + g.integers(1, 41, size=100).tolist() + [1]
    many = g.integers(1, 6, size=3000).tolist()          # more segments than the grid
    return [(256, mixed), (37, mixed), (1, [1, 2, 5]), (1000, [1, 7, 2500]), (40, many), (258, [1])]


@pytest.mark.parametrize("case", range(6))
def test_segment_mean_normalize(case):
    E, counts = _segment_cases()[case]
    R = sum(counts)
    g = torch.Generator().manual_seed(case)
    x_cpu = torch.randn(R, E, generator=g) + 0.1
    x = x_cpu.to(DEV).requires_grad_(True)
    y = tr.segment_mean_normalize(x, counts)
    x64 = x_cpu.double().requires_grad_(True)
    ref = mean_normalize64(x64, counts)
    assert y.shape == (len(counts), E)
    row_err = (y.detach().double().cpu() - ref.detach()).norm(dim=1).max().item()   # the rows are unit vectors
    assert row_err <= FWD_TOL, row_err
    y2 = tr.segment_mean_normalize(x.detach(), counts)
    assert torch.equal(y.detach(), y2)                    # fixed summation order

    w = torch.randn(len(counts), E, generator=g)
    (y * w.to(DEV)).sum().backward()
    (ref * w.double()).sum().backward()
    assert rel_err(x.grad, x64.grad) <= GRAD_TOL, rel_err(x.grad, x64.grad)
    gx = x.grad.clone()
    x.grad = None
    (tr.segment_mean_normalize(x, counts) * w.to(DEV)).sum().backward()
    assert torch.equal(x.grad, gx)


def test_embed_speakers_against_fp64():
    enc = _fixture_encoder("spkenc_tt_lstm_h64_L2")
    counts = [1, 4, 10, 2000] + _lengths(3, 200, 30)
    d = torch.nn.functional.normalize(torch.rand(sum(counts), 32, generator=torch.Generator().manual_seed(4)), dim=1)
    s = enc.embed_speakers(d.to(DEV), counts)
    assert s.shape == (len(counts), 32)
    assert (s.double().cpu() - mean_normalize64(d.double(), counts)).norm(dim=1).max().item() <= FWD_TOL


# ---- end to end --------------------------------------------------------------------------------------------------------------
CASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "spkenc_*.npz")))
KW = {"spkenc_tt_lstm_h64_L2": dict(compression="tt", n_cores=3, rank=4),
      "spkenc_dense_lstm_h128_L1": dict(compression=None),
      "spkenc_tt_gru_h64_L1": dict(compression="tt", n_cores=2, rank=2, use_gru=True)}
PROJ = {"proj_tt_lstm_h64_p16_L2": (64, 2, dict(compression="tt", n_cores=2, rank=4, proj_size=16)),
        "proj_dense_lstm_h256_p128_L1": (256, 1, dict(compression=None, proj_size=128))}


def _fixture_encoder(name):
    if name in PROJ:
        H, L, kw = PROJ[name]
        torch.manual_seed(6)
        with redirect_stdout(io.StringIO()):
            enc = tr.SpeakerEncoder(40, H, L, 32, CPU, None, **kw)
        return enc.to(DEV)
    g = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    _, _, _, H, L = (int(v) for v in g["shape"])
    with redirect_stdout(io.StringIO()):
        enc = tr.SpeakerEncoder(40, H, L, 32, CPU, None, **KW[name])
    enc.load_state_dict({k[len("param:"):]: torch.from_numpy(v) for k, v in g.items() if k.startswith("param:")})
    return enc.to(DEV)


@pytest.mark.parametrize("name", CASES + sorted(PROJ))
def test_embed_utterances_matches_the_composition(name):
    enc = _fixture_encoder(name)
    lengths = _lengths(5, 300, 3000, fixed=(1, 79, 160, 200, 281, 999))
    frames = torch.rand(sum(lengths), 40, generator=torch.Generator().manual_seed(7)).to(DEV)
    w = torch.randn(len(lengths), 32, generator=torch.Generator().manual_seed(8)).to(DEV)

    d = enc.embed_utterances(frames, lengths)
    assert d.shape == (len(lengths), 32)
    (d * w).sum().backward()
    grads = {k: p.grad.clone() for k, p in enc.named_parameters() if p.grad is not None}
    enc.zero_grad(set_to_none=True)

    utts = torch.split(frames, lengths)
    wins = [windows_of(u) for u in utts]
    emb = enc(torch.cat(wins))
    ref = mean_normalize64(emb, [x.shape[0] for x in wins])
    assert rel_err(d, ref) <= FWD_TOL, rel_err(d, ref)
    (ref * w.double()).sum().backward()
    ref_grads = {k: p.grad for k, p in enc.named_parameters() if p.grad is not None}
    expected = {k for k, _ in enc.named_parameters() if not k.startswith("similarity_")}
    assert set(grads) == set(ref_grads) == expected
    bad = {k: rel_err(grads[k], ref_grads[k]) for k in grads if not rel_err(grads[k], ref_grads[k]) <= GRAD_TOL}
    assert not bad, bad

    with torch.no_grad():
        d2 = enc.eval().embed_utterances(frames, lengths)
    assert rel_err(d2, d) <= FWD_TOL


def test_batch_independence():
    enc = _fixture_encoder("spkenc_tt_lstm_h64_L2").eval()
    lengths = _lengths(9, 500, 3000)
    frames = torch.rand(sum(lengths), 40, generator=torch.Generator().manual_seed(10)).to(DEV)
    with torch.no_grad():
        d = enc.embed_utterances(frames, lengths)
        off = np.cumsum([0] + lengths)
        for i in (0, 17, 499):
            alone = enc.embed_utterances(frames[off[i]:off[i + 1]], [lengths[i]])
            assert rel_err(alone[0], d[i]) <= FWD_TOL, (i, rel_err(alone[0], d[i]))
