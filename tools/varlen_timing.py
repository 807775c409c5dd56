"""Cost of variable-length rows (DESIGN.md §4.22).

    python tools/varlen_timing.py [--out DIR] [--reps 5] [--utterances 2620] [--seed 0]

1. Full-utterance embeddings: the cfg3 encoder (3 x TT-LSTM d3 r8, I 40, H 256, E 256), eval mode, under no_grad, on the
   synthetic utterance set of tools/utterance_embed_timing.py (log-normal lengths, median 700 frames, clipped to
   [100, 3500]).  full_call_ms: one embed_utterances(using_partials=False) call on device-resident packed frames (median of
   --reps); loop_ms: the reference family's full mode, forward on each utterance alone (one pass after a warm-up of 20);
   padded_fraction: the share of the call's row-steps past a row's length (every row runs max(lengths) steps).
2. Training step: TTLSTM(40, 256, 3, d3 r8) at B 640, T 160 (the cfg3 shape), forward + backward of out.sum() + h_n.sum()
   through forward_states, three ways alternated --reps times (medians): a PackedSequence of all lengths = T
   (packed_ms), the padded tensor with lengths all T through functional.rnn_sequence (padded_lengths_ms: the same
   engine call without torch's pad / pack copies), and the padded tensor without lengths (no_lengths_ms).  A
   torch.profiler pass over one packed step gives the share of the k_varlen_* kernels in its kernel time.
3. The same three ways for the dense LSTM(40, 256, 3) at B 640, T 160, whose backward masks each step's output gradient
   with one extra launch per step.
The card name and power limit are read in the same run.  One JSON object on stdout and, with --out, in
DIR/varlen_timing.json.  Needs a CUDA device.
"""
import argparse
import io
import json
import os
import sys
from contextlib import redirect_stdout

import numpy as np
import torch
from torch.nn.utils.rnn import pack_padded_sequence

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import tensorized_rnn_b200 as tr  # noqa: E402
from chunked_states import card_info  # noqa: E402
from utterance_embed_timing import lengths_of, timed  # noqa: E402


def step(m, x, mode, packed, lengths):
    if mode == "packed":
        out, (h, c) = m.forward_states(packed)
        out = out.data
    elif mode == "padded_lengths":
        if isinstance(m, tr.TTLSTM):
            out, h, c = tr.functional.rnn_sequence(m.spec(), x, None, None, m.flat_parameters(), layer_states=True,
                                                   lengths=lengths)
        else:
            out, h, c = m._run_padded(x, None, None, True, lengths)
    else:
        out, (h, c) = m.forward_states(x)
    (out.sum() + h.sum()).backward()


def step_times(m, x, reps):
    B, T = x.shape[:2]
    lengths = torch.full((B,), T)
    packed = pack_padded_sequence(x, lengths, batch_first=True)
    modes = ("packed", "padded_lengths", "no_lengths")
    for mode in modes:
        step(m, x, mode, packed, lengths)
    ms = {mode: [] for mode in modes}
    for _ in range(reps):
        for mode in modes:
            ms[mode].append(timed(lambda: step(m, x, mode, packed, lengths)))
    res = {mode + "_ms": float(np.median(v)) for mode, v in ms.items()}
    res.update({mode + "_ms_all": v for mode, v in ms.items()})
    return res, packed, lengths


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--utterances", type=int, default=2620)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    if args.out:
        os.makedirs(args.out, exist_ok=True)
    res = {"card": card_info()}

    torch.manual_seed(0)
    with redirect_stdout(io.StringIO()):
        enc = tr.SpeakerEncoder(40, 256, 3, 256, torch.device("cpu"), None, compression="tt", n_cores=3, rank=8)
    enc = enc.to(dev).eval()
    lengths = lengths_of(args.utterances, args.seed)
    frames = torch.rand(sum(lengths), 40, generator=torch.Generator().manual_seed(args.seed)).to(dev)
    utts = torch.split(frames, lengths)
    with torch.no_grad():
        d = enc.embed_utterances(frames, lengths, using_partials=False)
        torch.cuda.synchronize()
        call = [timed(lambda: enc.embed_utterances(frames, lengths, using_partials=False)) for _ in range(args.reps)]
        for u in utts[:20]:
            enc(u[None])
        ref = [None]
        loop = timed(lambda: ref.__setitem__(0, torch.cat([enc(u[None]) for u in utts])))
    res["full_utterance"] = {
        "utterances": len(lengths), "frames": int(sum(lengths)), "max_len": int(max(lengths)),
        "padded_fraction": 1.0 - sum(lengths) / (len(lengths) * max(lengths)),
        "full_call_ms": float(np.median(call)), "full_call_ms_all": call, "loop_ms": loop,
        "loop_over_call": loop / float(np.median(call)),
        "rel_diff_call_vs_loop": float((d - ref[0]).norm() / ref[0].norm())}

    torch.manual_seed(0)
    m = tr.TTLSTM(40, 256, 3, torch.device("cpu"), n_cores=3, tt_rank=8).to(dev)
    B, T = 640, 160
    x = torch.rand(B, T, 40, device=dev)
    tt, packed, lengths = step_times(m, x, args.reps)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step(m, x, "packed", packed, lengths)
        torch.cuda.synchronize()
    total = varlen = 0.0
    for ev in prof.key_averages():
        us = getattr(ev, "self_device_time_total", None)
        us = ev.self_cuda_time_total if us is None else us
        total += us
        if "k_varlen" in ev.key:
            varlen += us
    res["training_step"] = dict(tt, model="TTLSTM(40, 256, 3, n_cores=3, tt_rank=8), B 640, T 160, lengths all T",
                                varlen_kernel_share=varlen / total if total else None, kernel_ms_total=total / 1e3)
    torch.manual_seed(0)
    md = tr.LSTM(40, 256, 3, torch.device("cpu")).to(dev)
    dn, _, _ = step_times(md, x, args.reps)
    res["dense_training_step"] = dict(dn, model="LSTM(40, 256, 3) (dense), B 640, T 160, lengths all T")
    print(json.dumps(res))
    if args.out:
        with open(os.path.join(args.out, "varlen_timing.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
