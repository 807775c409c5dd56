"""Cost of utterance-level embeddings (`SpeakerEncoder.embed_utterances`, DESIGN.md §4.21) against the per-utterance loop of
Real-Time-Voice-Cloning's `embed_utterance`.

    python tools/utterance_embed_timing.py [--out DIR] [--reps 5] [--utterances 2620] [--seed 0]

Model: the cfg3 encoder (3 x TT-LSTM d3 r8, I 40, H 256, E 256), eval mode, under no_grad.  Input: --utterances synthetic
utterances (2 620 = the size of LibriSpeech test-clean) of uniform random frames; lengths drawn with numpy's
default_rng(--seed) from a log-normal with median 700 frames and sigma 0.6, rounded and clipped to [100, 3500] frames.
Timed with CUDA events after warm-up:
  batched_call_ms   one embed_utterances call on device-resident packed frames (median of --reps);
  batched_h2h_ms    the same call from host frames to host d-vectors (copy in, call, copy out; median of --reps);
  loop_ms           the reference family's loop: per utterance, windows sliced and zero-padded on the host, one copy to the
                    device, one enc(windows), the window embeddings copied back, averaged and normalised on the host (one
                    pass after a warm-up of 20 utterances).
A separate torch.profiler pass over one embed_utterances call gives each kernel's device time and its share of the call's
kernel time.  The card name and power limit are read in the same run (nvidia-smi).  Printed as one JSON object and, with
--out, written to DIR/utterance_embed_timing.json.  Needs a CUDA device; there is no CPU path.
"""
import argparse
import io
import json
import os
import sys
from contextlib import redirect_stdout

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import tensorized_rnn_b200 as tr  # noqa: E402
from chunked_states import card_info  # noqa: E402

P, OVERLAP, MIN_COVERAGE = 160, 0.5, 0.75


def lengths_of(n, seed):
    g = np.random.default_rng(seed)
    return np.clip(np.round(g.lognormal(np.log(700.0), 0.6, size=n)), 100, 3500).astype(np.int64).tolist()


def loop_embed(enc, utts_np, dev):
    """Real-Time-Voice-Cloning's embed_utterance, once per utterance: host slicing, one stack call, host mean."""
    out = []
    for u in utts_np:
        n = u.shape[0]
        starts = tr.partial_windows([n], P, OVERLAP, MIN_COVERAGE)[0]
        wins = np.zeros((len(starts), P, u.shape[1]), dtype=np.float32)
        for i, s in enumerate(starts):
            wins[i, :min(P, n - s)] = u[s:s + P]
        part = enc(torch.from_numpy(wins).to(dev)).cpu().numpy()
        m = part.mean(axis=0)
        out.append(m / np.linalg.norm(m))
    return np.stack(out)


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def kernel_shares(enc, frames, lengths, out_dir):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        enc.embed_utterances(frames, lengths)
        torch.cuda.synchronize()
    rows = []
    for ev in prof.key_averages():
        if getattr(ev, "device_type", None) is None or "CUDA" not in str(ev.device_type):
            continue
        us = getattr(ev, "self_device_time_total", None)
        if us is None:
            us = ev.self_cuda_time_total
        if us > 0:
            rows.append({"kernel": ev.key, "calls": ev.count, "ms": us / 1e3})
    total = sum(r["ms"] for r in rows)
    for r in rows:
        r["share"] = r["ms"] / total
    rows.sort(key=lambda r: -r["ms"])
    if out_dir:
        prof.export_chrome_trace(os.path.join(out_dir, "utterance_embed.pt.trace.json"))
    return {"kernel_ms_total": total, "kernels": rows}


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

    torch.manual_seed(0)
    with redirect_stdout(io.StringIO()):
        enc = tr.SpeakerEncoder(40, 256, 3, 256, torch.device("cpu"), None, compression="tt", n_cores=3, rank=8)
    enc = enc.to(dev).eval()
    lengths = lengths_of(args.utterances, args.seed)
    packed = torch.rand(sum(lengths), 40, generator=torch.Generator().manual_seed(args.seed)).numpy()
    frames = torch.from_numpy(packed).to(dev)
    utts_np = np.split(packed, np.cumsum(lengths)[:-1])
    k = tr.partial_windows(lengths, P, OVERLAP, MIN_COVERAGE)[2]

    res = {"card": card_info(), "model": "SpeakerEncoder(40, 256, 3, 256, compression='tt', n_cores=3, rank=8), eval",
           "utterances": len(lengths), "frames": int(sum(lengths)), "windows": int(k.sum()),
           "lengths": {"distribution": "round(lognormal(ln 700, 0.6)) clipped to [100, 3500], numpy default_rng(%d)" % args.seed,
                       "min": int(min(lengths)), "median": float(np.median(lengths)), "mean": float(np.mean(lengths)),
                       "max": int(max(lengths))}}
    with torch.no_grad():
        d = enc.embed_utterances(frames, lengths)                                  # warm-up
        torch.cuda.synchronize()
        call = [timed(lambda: enc.embed_utterances(frames, lengths)) for _ in range(args.reps)]
        h2h = [timed(lambda: enc.embed_utterances(torch.from_numpy(packed).to(dev), lengths).cpu()) for _ in range(args.reps)]
        loop_embed(enc, utts_np[:20], dev)                                          # warm-up
        ref = [None]
        loop = timed(lambda: ref.__setitem__(0, loop_embed(enc, utts_np, dev)))
        diff = float(np.linalg.norm(d.cpu().numpy() - ref[0]) / np.linalg.norm(ref[0]))
        res.update({"batched_call_ms": float(np.median(call)), "batched_call_ms_all": call,
                    "batched_h2h_ms": float(np.median(h2h)), "batched_h2h_ms_all": h2h, "loop_ms": loop,
                    "loop_over_batched_call": loop / float(np.median(call)),
                    "rel_diff_batched_vs_loop": diff})
        res["profile"] = kernel_shares(enc, frames, lengths, args.out)
    print(json.dumps(res))
    if args.out:
        with open(os.path.join(args.out, "utterance_embed_timing.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
