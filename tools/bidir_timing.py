"""Bidirectional stacks against unidirectional ones (`bidirectional=True`, DESIGN.md §4.17).

    python tools/bidir_timing.py [--out DIR] [--reps 7] [--warmup 2] [--batches 80,160,320,640] [--no-profile]

(a) ms per step, training (forward + backward, upstream gradient on every output) and inference (no_grad forward), for
    the cfg1 shape (TT-LSTM d2 r4, I 1, B 256, T 784, one layer), the cfg2 shape (TT-GRU d2 r4, I 1, B 1024, T 784, one
    layer) and the cfg3 shape (3 x TT-LSTM d3 r8, I 40, T 160) at each batch of --batches; the same module with
    bidirectional=False beside it and the ratio bidirectional / unidirectional.
(b) the direction-handling kernels' own time at the cfg3 shape, B 640 (CUDA events over 50 launches each, inputs of
    105-210 MB, larger than L2): the join (forward with y_rev, backward with both gradients) and the layer-0 time-reversed
    add (reverse only, and the input-gradient sum), with the bytes each must move and the achieved rate against the
    7.7 TB/s data-sheet bandwidth.
(c) unless --no-profile, a separate torch.profiler pass over one bidirectional training step and one inference forward
    per shape: the time the two directions' recurrent kernels (k_rnn_*) run at the same time, as a share of the shorter
    direction's recurrent-kernel time.
(d) describe_plan of layer 1 of the bidirectional cfg3 stack at B 640 (its ih input is 2H = 512).
Card name and power limit are read in the same run (nvidia-smi).  Everything is printed as one JSON object and, with
--out, written to DIR/bidir_timing.json.  Needs a CUDA device; there is no CPU path.
"""
import argparse
import ctypes as C
import io
import json
import os
import sys
import tempfile
from contextlib import redirect_stdout

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import tensorized_rnn_b200 as tr  # noqa: E402
from tensorized_rnn_b200 import _lib  # noqa: E402
from chunked_states import card_info, timed  # noqa: E402

HBM_TBPS = 7.7


def shapes(batches):
    out = [("cfg1", "lstm", 1, 256, 1, 2, 4, 256, 784), ("cfg2", "gru", 1, 256, 1, 2, 4, 1024, 784)]
    out += [("cfg3_B%d" % b, "lstm", 40, 256, 3, 3, 8, b, 160) for b in batches]
    return out


def module(cell, I, H, L, d, r, bidirectional, dev):
    torch.manual_seed(0)
    with redirect_stdout(io.StringIO()):
        m = (tr.TTLSTM if cell == "lstm" else tr.TTGRU)(I, H, L, torch.device("cpu"), n_cores=d, tt_rank=r,
                                                        bidirectional=bidirectional)
    return m.to(dev)


def step_fns(m, x, w):
    def train():
        for p in m.parameters():
            p.grad = None
        out = m(x)[0]
        (out * w).sum().backward()

    def infer():
        with torch.no_grad():
            m(x)
    return train, infer


def step_times(args, dev):
    res = {}
    for name, cell, I, H, L, d, r, B, T in shapes(args.batches):
        g = torch.Generator().manual_seed(1)
        x = torch.rand(B, T, I, generator=g).to(dev)
        ent = {"shape": "%s %s I=%d H=%d L=%d d=%d r=%d B=%d T=%d" % (name, cell, I, H, L, d, r, B, T)}
        for bi in (False, True):
            m = module(cell, I, H, L, d, r, bi, dev)
            w = torch.randn(B, T, (2 if bi else 1) * H, generator=g).to(dev)
            train, infer = step_fns(m, x, w)
            key = "bidirectional" if bi else "unidirectional"
            ent[key] = {"train_ms": timed(train, args.reps, args.warmup), "infer_ms": timed(infer, args.reps, args.warmup)}
            del m
            torch.cuda.empty_cache()
        for k in ("train_ms", "infer_ms"):
            ent["ratio_" + k[:-3]] = ent["bidirectional"][k] / ent["unidirectional"][k]
        res[name] = ent
        print(json.dumps({name: ent}), file=sys.stderr)
    return res


def kernel_times(dev, reps=50):
    """Own time of the direction-handling kernels at the cfg3 shape, B 640: T 160, H 256, I 40."""
    lib = _lib.load()
    B, T, H, I = 640, 160, 256, 40
    st = torch.cuda.current_stream(dev).cuda_stream
    f, r = torch.rand(B, T, H, device=dev), torch.rand(B, T, H, device=dev)
    y, yr = torch.empty(B, T, 2 * H, device=dev), torch.empty(B, T, 2 * H, device=dev)
    df, dr = torch.empty(B, T, H, device=dev), torch.empty(B, T, H, device=dev)
    x, xr, dx = torch.rand(B, T, I, device=dev), torch.rand(B, T, I, device=dev), torch.empty(B, T, I, device=dev)
    p = lambda t: C.c_void_p(t.data_ptr())                                  # noqa: E731
    n = B * T * H * 4
    m = B * T * I * 4
    cases = {
        "join_forward": (lambda: lib.ttrnn_bidir_join(B, T, H, 0, p(f), p(r), p(y), p(yr), st), 2 * n, 4 * n),
        "join_backward": (lambda: lib.ttrnn_bidir_join(B, T, H, 1, p(y), p(yr), p(df), p(dr), st), 4 * n, 2 * n),
        "reverse_input": (lambda: lib.ttrnn_time_reverse_add(B, T, I, None, p(x), p(xr), st), m, m),
        "input_grad_sum": (lambda: lib.ttrnn_time_reverse_add(B, T, I, p(x), p(xr), p(dx), st), 2 * m, m),
    }
    out = {"shape": "B=%d T=%d H=%d I=%d" % (B, T, H, I)}
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
        out[name] = {"us": ms * 1e3, "read_MB": rd / 1e6, "write_MB": wr / 1e6, "TB_per_s": tbps,
                     "share_of_7.7TB_per_s": tbps / HBM_TBPS}
    return out


def _union(iv):
    iv = sorted(iv)
    out = []
    for a, b in iv:
        if out and a <= out[-1][1]:
            out[-1][1] = max(out[-1][1], b)
        else:
            out.append([a, b])
    return out


def _intersect(u, v):
    i = j = 0
    tot = 0.0
    while i < len(u) and j < len(v):
        lo, hi = max(u[i][0], v[j][0]), min(u[i][1], v[j][1])
        tot += max(0.0, hi - lo)
        if u[i][1] < v[j][1]:
            i += 1
        else:
            j += 1
    return tot


def overlap(args, dev):
    """Recurrent-kernel (k_rnn_*) time per stream in one profiled bidirectional step, and how much of it overlaps."""
    from torch.profiler import ProfilerActivity, profile
    res = {}
    for name, cell, I, H, L, d, r, B, T in shapes([80, 640]):
        g = torch.Generator().manual_seed(1)
        x = torch.rand(B, T, I, generator=g).to(dev)
        m = module(cell, I, H, L, d, r, True, dev)
        w = torch.randn(B, T, 2 * H, generator=g).to(dev)
        train, infer = step_fns(m, x, w)
        for mode, fn in (("train", train), ("infer", infer)):
            fn()
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                fn()
                torch.cuda.synchronize()
            with tempfile.TemporaryDirectory() as tmp:
                path = os.path.join(tmp, "trace.json")
                prof.export_chrome_trace(path)
                with open(path) as fh:
                    ev = json.load(fh)["traceEvents"]
            per_stream = {}
            for e in ev:
                if e.get("cat") == "kernel" and "k_rnn_" in e.get("name", ""):
                    s = e.get("args", {}).get("stream")
                    per_stream.setdefault(s, []).append((float(e["ts"]), float(e["ts"]) + float(e["dur"])))
            streams = sorted(per_stream, key=lambda s: -len(per_stream[s]))
            ent = {"streams": {str(s): {"kernels": len(per_stream[s]),
                                        "busy_us": sum(b - a for a, b in _union(per_stream[s]))} for s in streams}}
            if len(streams) >= 2:
                u, v = _union(per_stream[streams[0]]), _union(per_stream[streams[1]])
                both = _intersect(u, v)
                shorter = min(sum(b - a for a, b in u), sum(b - a for a, b in v))
                ent["overlap_us"] = both
                ent["overlap_share_of_shorter_direction"] = both / shorter if shorter > 0 else 0.0
            res["%s_%s" % (name, mode)] = ent
        del m
        torch.cuda.empty_cache()
    return res


def plan_layer1(dev):
    m = module("lstm", 40, 256, 3, 3, 8, True, dev)
    return {c: _lib.describe_plan(getattr(m, c)._single_step_spec().desc(640, 160), training=True)
            for c in ("cell1", "cell1_reverse")}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--batches", default="80,160,320,640", help="batch sizes of the cfg3 shape")
    ap.add_argument("--no-profile", action="store_true")
    args = ap.parse_args()
    args.batches = [int(v) for v in args.batches.split(",") if v]
    if not torch.cuda.is_available():
        raise SystemExit("bidir_timing.py needs a CUDA device")
    dev = torch.device("cuda:0")
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi": card_info(), "plan_layer1_cfg3_B640": plan_layer1(dev),
           "kernels": kernel_times(dev), "steps": step_times(args, dev)}
    if not args.no_profile:
        res["overlap"] = overlap(args, dev)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bidir_timing.json"), "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
