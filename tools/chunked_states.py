"""A sequence run in pieces with per-layer states carried (`forward_states`, DESIGN.md §4.16), against one call.

    python tools/chunked_states.py [--out DIR] [--reps 5] [--warmup 2] [--chunks 40,16]

(a) inference, cfg4 shape (3 x TT-LSTM d4 r16, 16 384 utterances x 160 frames x 40 features): one 160-step call against
    160 / c calls of c steps each, every call seeded with the previous call's (L, B, H) final states -- the streaming
    case.  Reports ms per 160 frames, the per-call overhead (extra time / extra calls: planning, rank padding, the dense
    W_ih formed again per call) and the largest output and final-state difference.
(b) training, cfg3 shape (3 x TT-LSTM d3 r8, 640 x 160 x 40): one 160-step forward + backward against two 80-step calls
    linked through their states without detaching (truncated BPTT's building block).  Reports ms per training step and
    the largest norm-wise relative parameter-gradient difference.
Card name and power limit are read in the same run (nvidia-smi).  Everything is printed as one JSON object and, with
--out, written to DIR/chunked_states.json.  Needs a CUDA device; there is no CPU path.
"""
import argparse
import io
import json
import os
import subprocess
import sys
from contextlib import redirect_stdout

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import tensorized_rnn_b200 as tr  # noqa: E402


def card_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        res = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=60)
        return {"query": q, "value": res.stdout.strip()}
    except Exception as e:                      # reported, not fatal
        return {"query": q, "error": str(e)}


def module(I, H, L, d, r, dev):
    torch.manual_seed(0)
    with redirect_stdout(io.StringIO()):
        m = tr.TTLSTM(I, H, L, torch.device("cpu"), n_cores=d, tt_rank=r)
    return m.to(dev)


def timed(fn, reps, warmup):
    """Median milliseconds of fn() over `reps` runs (CUDA events, synchronised)."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    ms.sort()
    return ms[len(ms) // 2]


def rel(a, b):
    return float((a - b).double().norm() / b.double().norm())


def inference(args, dev):
    B, T, I, H, L = 16384, 160, 40, 256, 3
    m = module(I, H, L, 4, 16, dev)
    x = torch.rand(B, T, I, generator=torch.Generator().manual_seed(1)).to(dev)
    res = {"shape": "cfg4: 3 x TT-LSTM d4 r16, B=%d T=%d I=%d" % (B, T, I)}

    def chunked(c):
        states, outs = None, []
        for t0 in range(0, T, c):
            o, states = m.forward_states(x[:, t0:t0 + c], states)
            outs.append(o)
        return torch.cat(outs, dim=1), states

    with torch.no_grad():
        out1, (h1, c1) = m.forward_states(x)
        t1 = timed(lambda: m.forward_states(x), args.reps, args.warmup)
        res["one_call"] = {"calls": 1, "ms_per_160_frames": t1}
        for c in args.chunks:
            out, (h, cc) = chunked(c)
            tc = timed(lambda: chunked(c), args.reps, args.warmup)
            n = -(-T // c)
            res["chunks_of_%d" % c] = {
                "calls": n, "ms_per_160_frames": tc,
                "overhead_ms_per_extra_call": (tc - t1) / (n - 1) if n > 1 else 0.0,
                "max_abs_output_diff": float((out - out1).abs().max()), "rel_output_diff": rel(out, out1),
                "max_abs_final_state_diff": max(float((h - h1).abs().max()), float((cc - c1).abs().max())),
                "bitwise_equal": bool(torch.equal(out, out1) and torch.equal(h, h1) and torch.equal(cc, c1)),
            }
    return res


def training(args, dev):
    B, T, I, H, L = 640, 160, 40, 256, 3
    m = module(I, H, L, 3, 8, dev)
    g = torch.Generator().manual_seed(2)
    x = torch.rand(B, T, I, generator=g).to(dev)
    w = torch.randn(B, T, H, generator=g).to(dev)
    res = {"shape": "cfg3: 3 x TT-LSTM d3 r8, B=%d T=%d I=%d" % (B, T, I)}

    def step(pieces):
        for p in m.parameters():
            p.grad = None
        states, outs, c = None, [], T // pieces
        for t0 in range(0, T, c):
            o, states = m.forward_states(x[:, t0:t0 + c], states)
            outs.append(o)
        (torch.cat(outs, dim=1) * w).sum().backward()

    step(1)
    g1 = [p.grad.clone() for p in m.flat_parameters()]
    step(2)
    g2 = [p.grad.clone() for p in m.flat_parameters()]
    res["one_call"] = {"calls": 1, "ms_per_step": timed(lambda: step(1), args.reps, args.warmup)}
    res["two_linked_calls"] = {"calls": 2, "ms_per_step": timed(lambda: step(2), args.reps, args.warmup),
                               "max_rel_param_grad_diff": max(rel(a, b) for a, b in zip(g2, g1))}
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--chunks", default="40,16", help="chunk lengths of the inference comparison (steps)")
    args = ap.parse_args()
    args.chunks = [int(v) for v in args.chunks.split(",") if v]
    if not torch.cuda.is_available():
        raise SystemExit("chunked_states.py needs a CUDA device")
    dev = torch.device("cuda:0")
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi": card_info(),
           "inference": inference(args, dev), "training": training(args, dev)}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "chunked_states.json"), "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
