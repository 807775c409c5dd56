"""Snapshot of the kernel routes a build of the library takes, for comparing two builds.

    python tools/route_snapshot.py --root TREE --out FILE

imports tensorized_rnn_b200 from TREE (a source tree with the library built in it) and writes one JSON line per
(case, option setting): the describe text for training and inference, the three workspace sizes, the launch count of
one forward + backward step and its recurrent and GEMM launches in issue order (kind, rows per CTA, CTAs, rows, steps),
recorded with ttrnn_kernel_timing.  Two builds that route identically give identical files.  Needs a CUDA device.
"""
import argparse
import ctypes as C
import io
import json
import os
import sys
from contextlib import redirect_stdout

HERE = os.path.dirname(os.path.abspath(__file__))

# option settings, each applied on top of the defaults (the default of every option touched is restored afterwards)
SETTINGS = [{}, {"merge_cores": 0}, {"merge_cores": 2}, {"split_kept": 0}, {"row_plan": 0}, {"row_groups": 0},
            {"static_kernels": 0}, {"chunk_steps": 48}, {"save_u_bytes": 0}, {"bwd_overlap": 0}, {"dense_hh_dw": 0},
            {"static_rows_fwd": 2, "static_rows_bwd": 2}]
DEFAULTS = {"merge_cores": 1, "split_kept": 1, "row_plan": 1, "row_groups": 1, "static_kernels": 1, "chunk_steps": 0,
            "save_u_bytes": 16 << 30, "bwd_overlap": 1, "dense_hh_dw": 1, "static_rows_fwd": 0, "static_rows_bwd": 0}


def cases():
    sys.path.insert(1, os.path.dirname(HERE))
    from bench import CONFIGS
    out = []
    for cid in (1, 2, 3, 4, 5, 6, 8, 9):                 # cfg7 is the dense baseline: no TT routes
        c = CONFIGS[cid]
        out.append(("cfg%d" % cid, c["cell"], c["I"], c["H"], c["L"], c["d"], c["r"], c["B"], c["T"], False))
    c = CONFIGS[3]
    for B in (80, 160, 320, 480, 640):
        out.append(("cfg3_B%d" % B, "lstm", c["I"], c["H"], c["L"], c["d"], c["r"], B, c["T"], False))
    c = CONFIGS[1]
    out.append(("cfg1_dx", "lstm", 1, c["H"], c["L"], c["d"], c["r"], c["B"], c["T"], True))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", required=True)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.root))
    import torch
    import tensorized_rnn_b200 as tr
    from tensorized_rnn_b200 import _lib
    lib = _lib.load()
    dev = torch.device("cuda:0")

    def records():
        kms, kcnt = (C.c_double * 7)(), (C.c_int64 * 7)()
        lib.ttrnn_kernel_times(kms, kcnt)
        n = lib.ttrnn_kernel_launch_records(None, 0)
        buf = (C.c_double * (6 * max(n, 1)))()
        lib.ttrnn_kernel_launch_records(buf, n)
        return [[int(buf[6 * i + j]) for j in range(5)] for i in range(n)]

    with open(args.out, "w") as f:
        for name, cell, I, H, L, d, r, B, T, want_dx in cases():
            torch.manual_seed(0)
            cls = tr.TTLSTM if cell == "lstm" else tr.TTGRU
            with redirect_stdout(io.StringIO()):
                m = cls(I, H, L, torch.device("cpu"), n_cores=d, tt_rank=r).to(dev)
            x = torch.rand(B, T, I, device=dev, requires_grad=want_dx)
            desc = m.spec().desc(B, T)
            for setting in SETTINGS:
                for k, v in setting.items():
                    assert lib.ttrnn_set_option(k.encode(), v) == 0, k
                try:
                    rec = {"case": name, "setting": setting}
                    for training in (1, 0):
                        buf = C.create_string_buffer(16384)
                        assert lib.ttrnn_rnn_describe(C.byref(desc), training, buf, 16384) >= 0, _lib.last_error()
                        rec["describe%d" % training] = buf.value.decode()
                    ws = _lib.RnnWorkspace()
                    assert lib.ttrnn_rnn_workspace_bytes(C.byref(desc), C.byref(ws)) == 0, _lib.last_error()
                    rec["workspace"] = [ws.saved_bytes, ws.fwd_scratch_bytes, ws.bwd_scratch_bytes]
                    for p in m.parameters():
                        p.grad = None
                    torch.cuda.synchronize()
                    records()
                    lib.ttrnn_launch_count(1)
                    lib.ttrnn_kernel_timing(1)
                    try:
                        m(x)[0].sum().backward()
                        torch.cuda.synchronize()
                    finally:
                        lib.ttrnn_kernel_timing(0)
                    rec["launches"] = int(lib.ttrnn_launch_count(1))
                    rec["records"] = records()
                finally:
                    for k in setting:
                        lib.ttrnn_set_option(k.encode(), DEFAULTS[k])
                f.write(json.dumps(rec) + "\n")
                f.flush()
            del m, x
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
