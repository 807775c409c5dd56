"""Cost of the projected TT-LSTM (`proj_size`, DESIGN.md §4.19).

    python tools/proj_timing.py [--out DIR] [--reps 5] [--warmup 1] [--shapes ge2e,cfg3]

Per shape, ms of a training step (forward + backward, upstream gradient on the output) and of an inference forward
(no_grad), median of --reps with the variants alternating call by call in the same run:
  proj        TTLSTM(proj_size=P), d3 r8 (runtime-shape kernels k_rnn_fwd_proj / k_rnn_bwd_proj);
  unproj_rt   TTLSTM at the same H without projection on the runtime-shape kernels (static_kernels = 0);
  torch       torch.nn.LSTM(proj_size=P, batch_first=True), FP32 (cuDNN).
Shapes: ge2e  the GE2E LSTMP shape, 3 layers, I 40, H 768, P 256, B 640, T 160;
        cfg3  3 layers, I 40, H 256, P 128, B 640, T 160.
Card name and power limit are read in the same run (nvidia-smi).  Printed as one JSON object and, with --out, written to
DIR/proj_timing.json.  Needs a CUDA device; there is no CPU path.
"""
import argparse
import io
import json
import os
import sys
from contextlib import redirect_stdout

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import tensorized_rnn_b200 as tr  # noqa: E402
from tensorized_rnn_b200 import _lib  # noqa: E402
from chunked_states import card_info  # noqa: E402

SHAPES = {"ge2e": dict(L=3, I=40, H=768, P=256, B=640, T=160), "cfg3": dict(L=3, I=40, H=256, P=128, B=640, T=160)}


def quiet(cls, *a, **k):
    torch.manual_seed(0)
    with redirect_stdout(io.StringIO()):
        return cls(*a, **k)


def with_static(value, fn):
    """fn run with the static_kernels option set to `value` (the plan is stamped at the forward, so the backward follows)."""
    lib = _lib.load()

    def run():
        lib.ttrnn_set_option(b"static_kernels", value)
        try:
            fn()
        finally:
            lib.ttrnn_set_option(b"static_kernels", 1)
    return run


def alternate(variants, reps, warmup):
    """{name: median ms} per variant, the variants interleaved call by call."""
    for fn in variants.values():
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in variants}
    for _ in range(reps):
        for k, fn in variants.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ms[k].append(a.elapsed_time(b))
    return {k: sorted(v)[len(v) // 2] for k, v in ms.items()}


def shape_run(s, args, dev):
    L, I, H, P, B, T = s["L"], s["I"], s["H"], s["P"], s["B"], s["T"]
    g = torch.Generator().manual_seed(1)
    x = torch.rand(B, T, I, generator=g).to(dev)
    wp = torch.randn(B, T, P, generator=g).to(dev)
    wh = torch.randn(B, T, H, generator=g).to(dev)
    proj = quiet(tr.TTLSTM, I, H, L, torch.device("cpu"), n_cores=3, tt_rank=8, proj_size=P).to(dev)
    plain = quiet(tr.TTLSTM, I, H, L, torch.device("cpu"), n_cores=3, tt_rank=8).to(dev)
    ref = torch.nn.LSTM(I, H, L, batch_first=True, proj_size=P).to(dev)

    def train(m, w):
        def fn():
            for p in m.parameters():
                p.grad = None
            (m(x)[0] * w).sum().backward()
        return fn

    def infer(m):
        def fn():
            with torch.no_grad():
                m(x)
        return fn

    training = alternate({"proj": train(proj, wp), "unproj_rt": with_static(0, train(plain, wh)),
                          "torch": train(ref, wp)}, args.reps, args.warmup)
    inference = alternate({"proj": infer(proj), "unproj_rt": with_static(0, infer(plain)), "torch": infer(ref)},
                          args.reps, args.warmup)
    return dict(shape=s, params=dict(proj=proj.param_count(), unproj=plain.param_count(),
                                     torch=sum(p.numel() for p in ref.parameters())),
                train_ms=training, infer_ms=inference,
                proj_over_unproj_rt=dict(train=training["proj"] / training["unproj_rt"],
                                         infer=inference["proj"] / inference["unproj_rt"]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--shapes", default="ge2e,cfg3")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("proj_timing.py needs a CUDA device (there is no CPU path)")
    dev = torch.device("cuda:0")
    res = dict(card=card_info(), reps=args.reps, warmup=args.warmup,
               shapes={name: shape_run(SHAPES[name], args, dev) for name in args.shapes.split(",")})
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "proj_timing.json"), "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
