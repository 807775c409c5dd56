"""Cost of the projected dense LSTM (`LSTM(proj_size=P)`, DESIGN.md §4.20) next to the projected TT-LSTM (§4.19).

    python tools/dense_proj_timing.py [--out DIR] [--reps 5] [--warmup 1]

At the GE2E LSTMP shape (3 layers, I 40, H 768, P 256, B 640, T 160), ms of a training step (forward + backward, upstream
gradient on the output) and of an inference forward (no_grad), median of --reps with the variants alternating call by
call in the same run:
  dense_proj  LSTM(proj_size=P), this engine's dense sequence call;
  tt_proj     TTLSTM(proj_size=P), d3 r8 (runtime-shape kernels k_rnn_fwd_proj / k_rnn_bwd_proj);
  dense       LSTM at the same H without projection;
  torch       torch.nn.LSTM(proj_size=P, batch_first=True), FP32 (cuDNN).
Also reports the norm-wise relative difference of dense_proj's output from torch.nn.LSTM(proj_size=P) with the same
weights (cuDNN with TF32 disabled for that comparison).  Card name and power limit are read in the same run
(nvidia-smi).  Printed as one JSON object and, with --out, written to DIR/dense_proj_timing.json.  Needs a CUDA device;
there is no CPU path.
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import tensorized_rnn_b200 as tr  # noqa: E402
from chunked_states import card_info  # noqa: E402
from proj_timing import alternate, quiet  # noqa: E402

SHAPE = dict(L=3, I=40, H=768, P=256, B=640, T=160)


def torch_copy(m, dev):
    """torch.nn.LSTM(proj_size) with the weights of dense LSTM m (ih bias zero: the dense cell has none)."""
    t = torch.nn.LSTM(m.input_size, m.hidden_size, m.num_layers, batch_first=True, proj_size=m.proj_size).to(dev)
    with torch.no_grad():
        for l in range(m.num_layers):
            c = getattr(m, "cell%d" % l)
            getattr(t, "weight_ih_l%d" % l).copy_(c.input_weights.weight)
            getattr(t, "weight_hh_l%d" % l).copy_(c.hidden_weights.weight)
            getattr(t, "bias_ih_l%d" % l).zero_()
            getattr(t, "bias_hh_l%d" % l).copy_(c.hidden_weights.bias)
            getattr(t, "weight_hr_l%d" % l).copy_(c.projection_weights.weight)
    return t


def run(args, dev):
    s = SHAPE
    L, I, H, P, B, T = s["L"], s["I"], s["H"], s["P"], s["B"], s["T"]
    g = torch.Generator().manual_seed(1)
    x = torch.rand(B, T, I, generator=g).to(dev)
    wp = torch.randn(B, T, P, generator=g).to(dev)
    wh = torch.randn(B, T, H, generator=g).to(dev)
    dense_proj = quiet(tr.LSTM, I, H, L, torch.device("cpu"), proj_size=P).to(dev)
    tt_proj = quiet(tr.TTLSTM, I, H, L, torch.device("cpu"), n_cores=3, tt_rank=8, proj_size=P).to(dev)
    dense = quiet(tr.LSTM, I, H, L, torch.device("cpu")).to(dev)
    ref = torch_copy(dense_proj, dev)

    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    with torch.no_grad():
        a, b = dense_proj(x)[0].double(), ref(x)[0].double()
    torch.backends.cudnn.allow_tf32 = tf32
    rel = float((a - b).norm() / b.norm())

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

    training = alternate({"dense_proj": train(dense_proj, wp), "tt_proj": train(tt_proj, wp), "dense": train(dense, wh),
                          "torch": train(ref, wp)}, args.reps, args.warmup)
    inference = alternate({"dense_proj": infer(dense_proj), "tt_proj": infer(tt_proj), "dense": infer(dense),
                           "torch": infer(ref)}, args.reps, args.warmup)
    return dict(shape=s, params=dict(dense_proj=dense_proj.param_count(), tt_proj=tt_proj.param_count(),
                                     dense=dense.param_count()),
                train_ms=training, infer_ms=inference, dense_proj_out_rel_vs_torch_fp32=rel,
                dense_proj_over_dense=dict(train=training["dense_proj"] / training["dense"],
                                           infer=inference["dense_proj"] / inference["dense"]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dense_proj_timing.py needs a CUDA device (there is no CPU path)")
    dev = torch.device("cuda:0")
    res = dict(card=card_info(), reps=args.reps, warmup=args.warmup, ge2e=run(args, dev))
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "dense_proj_timing.json"), "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
