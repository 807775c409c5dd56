"""Cost of inter-layer dropout (`dropout=p`, DESIGN.md §4.18).

    python tools/dropout_timing.py [--out DIR] [--reps 9] [--warmup 2] [--p 0.1]

(a) ms per training step (forward + backward, upstream gradient on the output), median of --reps, the variants of one
    scenario alternating step by step in the same run:
      cfg3        3 x TT-LSTM d3 r8, I 40, H 256, B 640, T 160: dropout 0 and dropout p in one stack call;
      workaround  the same three layers as three one-layer TTLSTM modules with torch.nn.functional.dropout between them
                  (what a user had to write before), p;
      cfg3_bidir  the cfg3 shape with bidirectional=True: dropout 0 and p;
      dense       dense LSTM, 3 layers, I 128, H 256, B 640, T 160: dropout 0 (one multi-layer call) and p (one-layer
                  calls with the mask kernel between them).
(b) the mask kernel's own time at the cfg3 boundary shape (B 640, T 160, F 256 and 512; CUDA events over 50 launches,
    105-210 MB per operand, larger than L2): forward, forward with the time-reversed copy, backward in place, with the
    bytes each moves and the rate against the 7.7 TB/s data-sheet bandwidth.
Card name and power limit are read in the same run (nvidia-smi).  Printed as one JSON object and, with --out, written to
DIR/dropout_timing.json.  Needs a CUDA device; there is no CPU path.
"""
import argparse
import ctypes as C
import io
import json
import os
import sys
from contextlib import redirect_stdout

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import tensorized_rnn_b200 as tr  # noqa: E402
from tensorized_rnn_b200 import _lib  # noqa: E402
from chunked_states import card_info  # noqa: E402

HBM_TBPS = 7.7
B, T, I, H = 640, 160, 40, 256


def quiet(cls, *a, **k):
    torch.manual_seed(0)
    with redirect_stdout(io.StringIO()):
        return cls(*a, **k)


def train_step(forward, params, x, w):
    def fn():
        for p in params:
            p.grad = None
        out = forward(x)
        (out * w).sum().backward()
    return fn


def alternate(variants, reps, warmup):
    """{name: median ms} of one training step per variant, the variants interleaved step by step."""
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


def with_dropout(m, p):
    def fwd(x):
        m.dropout = p
        return m(x)[0]
    return fwd


def scenarios(args, dev):
    g = torch.Generator().manual_seed(1)
    x = torch.rand(B, T, I, generator=g).to(dev)
    w = torch.randn(B, T, H, generator=g).to(dev)
    w2 = torch.randn(B, T, 2 * H, generator=g).to(dev)
    res = {}

    m = quiet(tr.TTLSTM, I, H, 3, torch.device("cpu"), n_cores=3, tt_rank=8).to(dev)
    layers = [quiet(tr.TTLSTM, I if l == 0 else H, H, 1, torch.device("cpu"), n_cores=3, tt_rank=8).to(dev)
              for l in range(3)]
    for l, one in enumerate(layers):                    # the same parameters as the stack
        one.cell0.load_state_dict(getattr(m, "cell%d" % l).state_dict())
    layer_params = [p for one in layers for p in one.parameters()]

    def workaround(x_):
        z = x_
        for l, one in enumerate(layers):
            z = one(z)[0]
            if l < 2:
                z = F.dropout(z, args.p, True)
        return z

    t = alternate({"dropout_0": train_step(with_dropout(m, 0.0), list(m.parameters()), x, w),
                   "dropout_p": train_step(with_dropout(m, args.p), list(m.parameters()), x, w),
                   "workaround": train_step(workaround, layer_params, x, w)}, args.reps, args.warmup)
    t["overhead_pct"] = 100 * (t["dropout_p"] / t["dropout_0"] - 1)
    t["workaround_vs_stack_pct"] = 100 * (t["workaround"] / t["dropout_p"] - 1)
    res["cfg3"] = t
    print(json.dumps({"cfg3": t}), file=sys.stderr)
    del m, layers, layer_params
    torch.cuda.empty_cache()

    mb = quiet(tr.TTLSTM, I, H, 3, torch.device("cpu"), n_cores=3, tt_rank=8, bidirectional=True).to(dev)
    t = alternate({"dropout_0": train_step(with_dropout(mb, 0.0), list(mb.parameters()), x, w2),
                   "dropout_p": train_step(with_dropout(mb, args.p), list(mb.parameters()), x, w2)}, args.reps, args.warmup)
    t["overhead_pct"] = 100 * (t["dropout_p"] / t["dropout_0"] - 1)
    res["cfg3_bidir"] = t
    print(json.dumps({"cfg3_bidir": t}), file=sys.stderr)
    del mb
    torch.cuda.empty_cache()

    xd = torch.rand(B, T, 128, generator=g).to(dev)
    md = quiet(tr.LSTM, 128, H, 3, torch.device("cpu")).to(dev)
    t = alternate({"dropout_0": train_step(with_dropout(md, 0.0), list(md.parameters()), xd, w),
                   "dropout_p": train_step(with_dropout(md, args.p), list(md.parameters()), xd, w)}, args.reps, args.warmup)
    t["overhead_pct"] = 100 * (t["dropout_p"] / t["dropout_0"] - 1)
    res["dense_lstm"] = t
    print(json.dumps({"dense_lstm": t}), file=sys.stderr)
    return res


def kernel_times(args, dev, reps=50):
    lib = _lib.load()
    st = torch.cuda.current_stream(dev).cuda_stream
    dp = _lib.Dropout(args.p, 0, 1, 0)
    p = lambda t: C.c_void_p(t.data_ptr())                                  # noqa: E731
    out = {}
    for Fw in (H, 2 * H):
        x, y, yr = (torch.rand(B, T, Fw, device=dev) for _ in range(3))
        n = B * T * Fw * 4
        cases = {
            "forward": (lambda: lib.ttrnn_dropout_apply(B, T, Fw, 0, 0, 0, C.byref(dp), p(x), p(y), None, st), n, n),
            "forward_with_reversed_copy": (lambda: lib.ttrnn_dropout_apply(B, T, Fw, 0, 0, 0, C.byref(dp), p(x), p(y),
                                                                           p(yr), st), n, 2 * n),
            "backward_in_place": (lambda: lib.ttrnn_dropout_apply(B, T, Fw, 0, 0, 1, C.byref(dp), p(y), p(y), None, st),
                                  n, n),
        }
        ent = {}
        for name, (fn, rd, wr) in cases.items():
            for _ in range(3):
                _lib.check(fn(), name)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                fn()
            b.record()
            torch.cuda.synchronize()
            ms = a.elapsed_time(b) / reps
            tbps = (rd + wr) / (ms * 1e-3) / 1e12
            ent[name] = {"us": ms * 1e3, "read_MB": rd / 1e6, "write_MB": wr / 1e6, "TB_per_s": tbps,
                         "fraction_of_7.7TBps": tbps / HBM_TBPS}
        out["B=%d T=%d F=%d" % (B, T, Fw)] = ent
        del x, y, yr
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--p", type=float, default=0.1)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dropout_timing needs a CUDA device")
    dev = torch.device("cuda:0")
    res = {"card": card_info(), "p": args.p, "reps": args.reps,
           "kernel": kernel_times(args, dev), "steps": scenarios(args, dev)}
    res["card_after"] = card_info()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "dropout_timing.json"), "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
