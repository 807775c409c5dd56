#!/usr/bin/env python
"""Benchmark of the TT-LSTM / TT-GRU recurrence path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--configs 1,2,3,4,5] [--headline 3]
                    [--dump-outputs DIR]

Metric (BASELINE.json): TT-LSTM cell-steps/sec = batch x T / seconds of one forward(+backward) pass over the whole
stack.  One "step" = one such pass over one batch of synthetic input of the config's shape.

ONE JSON line (rank 0).  Top level = the HEADLINE workload: BASELINE.json configs[2], the GE2E speaker-encoder
training config (3 x TT-LSTM d3 r8, H 256, 40 mel, 64 speakers x 10 utterances = 640 sequences, T 160, fwd+bwd) --
the config north_star's scaling target names.  `all_configs` carries one record per BASELINE config (1..5) measured
in the same invocation: ms_per_step, value, e2e, per-kernel-group times, roofline, and at N = 1 a CPU baseline.

Scaling: `--gpus N` splits each config's GLOBAL batch evenly over the N ranks (SURVEY.md 8d) -> "scaling": "strong";
the weak-scaling figure (every rank runs the config's full batch) is measured beside it and reported as `weak`.
Training steps all-reduce the TT-core / bias gradients with NCCL inside the timed region.

`value` = device-resident throughput (CUDA events around each step, L2 flushed between steps, max over ranks);
`e2e` = the same pass through the public module API from pinned HOST input, with the H2D copy and a D2H read of the
result inside the timed region; `roofline` = the dominant kernel group against the FP32 FFMA peak measured live by an
FFMA probe kernel (MEASURED_PEAKS.json has no FP32 figure), in ALGORITHMIC FLOPs of the reference's core-by-core
sweep; `cpu_baseline` / `--impl reference` = the CPU oracle (a restatement of the reference's PyTorch path; the
reference itself cannot travel to the GPU box) on the host cores, on a bounded sample whose batch is stated.
"""
from __future__ import annotations

import argparse
import ctypes as C
import io
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from contextlib import redirect_stdout

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# name, cell, I, H, L, d, r, GLOBAL batch B, T, mode, upstream gradient, input kind, seed
CONFIGS = {
    1: dict(name="cfg1 sequential-MNIST TT-LSTM d2 r4", cell="lstm", I=1, H=256, L=1, d=2, r=4, B=256, T=784,
            mode="fwd+bwd", grad="out_last", inp="digits", seed=1111),
    2: dict(name="cfg2 permuted-MNIST TT-GRU d2 r4", cell="gru", I=1, H=256, L=1, d=2, r=4, B=1024, T=784,
            mode="fwd+bwd", grad="out_last", inp="digits_perm", seed=1111),
    3: dict(name="cfg3 GE2E speaker encoder 3xTT-LSTM d3 r8 (64 spk x 10 utt)", cell="lstm", I=40, H=256, L=3, d=3, r=8,
            B=640, T=160, mode="fwd+bwd", grad="hT", inp="uniform", seed=11),
    4: dict(name="cfg4 speaker encoder inference 3xTT-LSTM d4 r16 (16k utterances)", cell="lstm", I=40, H=256, L=3, d=4,
            r=16, B=16384, T=160, mode="fwd", grad=None, inp="uniform", seed=11),
    5: dict(name="cfg5 TT-LSTM H1024 d4 r8 sweep", cell="lstm", I=256, H=1024, L=1, d=4, r=8, B=4096, T=2000,
            mode="fwd+bwd", grad="dense", inp="uniform", seed=11),
    # secondary point SURVEY.md 8(a) asks for: the reference's own default GE2E model (params_model.py: d2, r2)
    6: dict(name="cfg3-alt GE2E speaker encoder 3xTT-LSTM d2 r2 (params_model.py defaults)", cell="lstm", I=40, H=256, L=3,
            d=2, r=2, B=640, T=160, mode="fwd+bwd", grad="hT", inp="uniform", seed=11),
    # the reference's own default GE2E model and batch (encoder/params_model.py: hidden 768, 1 layer, n_cores 2, rank 2,
    # 16 speakers x 32 utterances): rank-padded onto the static H = 768 kernels
    8: dict(name="ge2e-default GE2E speaker encoder 1xTT-LSTM H768 d2 r2 (params_model.py: 16 spk x 32 utt)", cell="lstm", I=40,
            H=768, L=1, d=2, r=2, B=512, T=160, mode="fwd+bwd", grad="hT", inp="uniform", seed=11),
    # cfg3 as the reference's training step actually runs it (encoder/main.py:271-290): recurrent stack -> TT projection ->
    # ReLU + L2 norm -> GE2E similarity matrix + softmax loss -> backward, with the head on the DEVICE (the reference moves the
    # embeddings to the CPU for the loss); same B x T units as cfg3
    9: dict(name="cfg3-step full GE2E training step: 3xTT-LSTM d3 r8 + TT projection + GE2E loss on the device", cell="lstm", I=40,
            H=256, L=3, d=3, r=8, B=640, T=160, mode="fwd+bwd", grad="ge2e", inp="uniform", seed=11, ge2e=(64, 10, 256)),
    # dense baseline of cfg3 through the same engine (SpeakerEncoder(compression=None), speaker_encoder.py:29-36): the paper's
    # dense-vs-TT comparison on one device path
    7: dict(name="cfg3-dense GE2E speaker encoder 3xLSTM (dense baseline)", cell="lstm", I=40, H=256, L=3, d=0, r=0, B=640, T=160,
            mode="fwd+bwd", grad="hT", inp="uniform", seed=11, dense=True),
}
# per-config (warmup, steps) when --warmup / --steps are not given (3 / 10 otherwise): cfg5 moves ~100 GB per step.
# Given on the command line, --warmup / --steps apply to every config.
STEP_DEFAULT = {5: (3, 3), 4: (3, 5)}
# --dump-outputs: an output array with more elements than this is written as a fixed, seeded sample of this many elements;
# all the arrays of one run together stay under DUMP_BYTES
DUMP_ELEMS = 1 << 18
DUMP_BYTES = 64 << 20
# CPU sample (batch, T) per config for the in-line cpu_baseline: about 5-15 s of CPU work each
CPU_SAMPLE = {1: (64, 784), 2: (64, 784), 3: (96, 160), 4: (32, 160), 5: (8, 200), 6: (96, 160), 7: (96, 160), 8: (96, 160), 9: (96, 160)}
KINDS = ["k_ttlinear_fwd", "k_rnn_fwd", "k_rnn_bwd", "k_ttlinear_bwd", "gemm_ih_fwd", "gemm_dx", "gemm_dw"]


# ------------------------------------------------------------------------------------------
def chain_flops(in_modes, out_modes, ranks):
    """FLOPs per row of the right-to-left TT sweep (SURVEY.md section 8d): sum_k 2 * M_k * K_k * N_k."""
    d = len(in_modes)
    total = 0
    for k in range(d):
        m = int(np.prod(out_modes[k + 1:])) * int(np.prod(in_modes[:k]))
        total += 2 * m * (in_modes[k] * ranks[k + 1]) * (out_modes[k] * ranks[k])
    return total


def algorithmic_flops(cfg):
    """Forward FLOPs per sequence-step: whole stack, hh chain of one layer, list of per-layer ih chains."""
    from tensorized_rnn_b200.shapes import tt_shape
    G = 4 if cfg["cell"] == "lstm" else 3
    H, d, r = cfg["H"], cfg["d"], cfg["r"]
    if cfg.get("dense"):
        hh = 2 * G * H * H
        ih = [2 * G * H * (cfg["I"] if l == 0 else H) for l in range(cfg["L"])]
        gate = 2 * G * H + 12 * H
        return sum(ih) + cfg["L"] * (hh + gate), hh, ih, gate
    ranks = [1] + [r] * (d - 1) + [1]
    hh = chain_flops(*tt_shape(H, H, d, G), ranks)
    ih = [chain_flops(*tt_shape(cfg["I"] if l == 0 else H, H, d, G), ranks) for l in range(cfg["L"])]
    gate = 2 * G * H + 12 * H
    return sum(ih) + cfg["L"] * (hh + gate), hh, ih, gate


def make_input(cfg, B, device="cpu"):
    g = torch.Generator().manual_seed(cfg["seed"])
    x = torch.rand(B, cfg["T"], cfg["I"], generator=g)
    if cfg["inp"].startswith("digits"):
        x = (x - 0.1307) / 0.3081                      # reference digit_classification/utils.py:9-10
    if cfg["inp"] == "digits_perm":
        np.random.seed(cfg["seed"])
        perm = torch.from_numpy(np.random.permutation(cfg["T"]))   # pmnist_test.py:92,132,154
        x = x[:, perm, :].contiguous()
    return x.to(device)


def upstream(cfg, out, hT):
    """Scalar whose gradient is the config's upstream gradient pattern."""
    if cfg["grad"] == "out_last":
        return out[:, -1, :].sum()
    if cfg["grad"] in ("hT", "ge2e"):         # CPU baseline of the GE2E step: the recurrent stack with a gradient on h_T
        return hT.sum()                          # (the head is a few ms on the CPU as well and is left out of the CPU figure)
    return None


class ClockSampler(object):
    """SM clock / power / throttle reasons sampled in-process through NVML for the whole run; `summary(windows)` keeps
    the samples that fall inside the timed regions.  Falls back to an nvidia-smi subprocess when pynvml is missing."""
    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, gpu_index, period=0.02):
        self.idx, self.period = gpu_index, period
        self.samples = []                    # (t, sm_mhz, max_mhz, power_w, reasons bitmask)
        self.stop_ev = threading.Event()
        self.thread = None
        self.source = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # honour CUDA_VISIBLE_DEVICES: NVML indexes physical devices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = self.idx
            if vis:
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if self.idx < len(ids) and ids[self.idx].isdigit():
                    phys = int(ids[self.idx])
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)

            def loop():
                while not self.stop_ev.is_set():
                    try:
                        sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                        pw = pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0
                        try:
                            rs = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                        except Exception:
                            rs = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                        self.samples.append((time.perf_counter(), float(sm), float(mx), pw, int(rs)))
                    except Exception:
                        pass
                    time.sleep(self.period)
            self.source = "nvml"
            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            pass
        try:
            q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                 "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
            proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "50",
                                     "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.proc = proc

            def loop():
                for ln in proc.stdout:
                    p = [v.strip() for v in ln.split(",")]
                    try:
                        rs = 0
                        for bit, v in zip((0x8, 0x40, 0x20, 0x4), p[3:7]):
                            if v.lower().startswith("active"):
                                rs |= bit
                        self.samples.append((time.perf_counter(), float(p[0]), float(p[1]), float(p[2]), rs))
                    except Exception:
                        continue
            self.source = "nvidia-smi"
            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
        except Exception:
            self.source = None

    def stop(self):
        self.stop_ev.set()
        if getattr(self, "proc", None) is not None:
            self.proc.terminate()

    def summary(self, windows):
        if self.source is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"], "samples": 0}
        ins = [s for s in self.samples if any(a <= s[0] <= b for a, b in windows)]
        reasons = sorted(k for k, bit in self.BAD.items() if any(s[4] & bit for s in ins))
        return {"sm_mhz": statistics.median(s[1] for s in ins) if ins else None,
                "sm_max_mhz": max(s[2] for s in ins) if ins else (self.samples[0][2] if self.samples else None),
                "power_w_max": max(s[3] for s in ins) if ins else None, "samples": len(ins),
                "samples_total": len(self.samples), "source": self.source, "reasons": reasons}


# ------------------------------------------------------------------------------------------
def run_cpu_oracle(cfg, B, T, steps, warmup):
    """Time the CPU oracle (restatement of the reference's PyTorch path) on the host cores."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ttrnn_oracle as oracle                      # bench: cpu_baseline / reference arm only
    torch.set_num_threads(os.cpu_count() or 1)
    c = dict(cfg)
    c["T"] = T
    if cfg.get("dense"):
        return run_cpu_dense_oracle(c, B, T, steps, warmup)
    layers = oracle.random_layers(cfg["cell"], cfg["I"], cfg["H"], cfg["L"], cfg["d"], cfg["r"], bias=True,
                                  seed=cfg["seed"], requires_grad=(cfg["mode"] != "fwd"))
    x = make_input(c, B)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        if cfg["mode"] == "fwd":
            with torch.no_grad():
                if cfg["cell"] == "lstm":
                    oracle.lstm_forward(layers, x)
                else:
                    oracle.gru_forward(layers, x)
        else:
            for p in oracle.flat_params(layers):
                p.grad = None
            if cfg["cell"] == "lstm":
                out, (h, _) = oracle.lstm_forward(layers, x)
            else:
                out, h = oracle.gru_forward(layers, x)
            loss = upstream(cfg, out, h)
            if loss is None:
                gd = torch.Generator().manual_seed(5)
                loss = (out * torch.rand(out.shape, generator=gd)).sum()
            loss.backward()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    sec = sum(times) / len(times)
    return B * T / sec, sec


def run_cpu_dense_oracle(cfg, B, T, steps, warmup):
    import dense_oracle                                # bench: cpu_baseline leg only
    import tensorized_rnn_b200 as tr
    torch.manual_seed(cfg["seed"])
    m = (tr.LSTM if cfg["cell"] == "lstm" else tr.GRU)(cfg["I"], cfg["H"], cfg["L"], torch.device("cpu"))
    layers = dense_oracle.layers_from_state_dict(m.state_dict(), cfg["L"], requires_grad=(cfg["mode"] != "fwd"))
    x = make_input(cfg, B)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        for p in dense_oracle.flat_params(layers):
            p.grad = None
        if cfg["cell"] == "lstm":
            out, (h, _) = dense_oracle.lstm_forward(layers, x)
        else:
            out, h = dense_oracle.gru_forward(layers, x)
        if cfg["mode"] != "fwd":
            upstream(cfg, out, h).backward()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    sec = sum(times) / len(times)
    return B * T / sec, sec


def config_json(cfg, B_rank, world, scaling):
    return {"workload": cfg["name"], "cell": cfg["cell"], "input_size": cfg["I"], "hidden_size": cfg["H"],
            "num_layers": cfg["L"], "n_cores": cfg["d"], "tt_rank": cfg["r"], "batch_per_gpu": B_rank,
            "global_batch": B_rank * world, "seq_len": cfg["T"], "mode": cfg["mode"], "upstream_grad": cfg["grad"],
            "parallelism": "dp%d (batch-sharded replicas, %s scaling)" % (world, scaling),
            "l2": "flushed between timed steps (256 MiB write)"}


# ------------------------------------------------------------------------------------------
class GpuBench(object):
    def __init__(self, rank, world, local_rank):
        import tensorized_rnn_b200 as tr
        from tensorized_rnn_b200 import _lib
        self.tr, self._lib = tr, _lib
        self.rank, self.world = rank, world
        torch.cuda.set_device(local_rank)
        self.dev = torch.device("cuda", local_rank)
        self.dist = None
        if world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)
            self.dist = dist
        self.lib = _lib.load()
        self.flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)
        self.windows = []                              # host-time windows of the timed regions (clock sampling)
        self.dumped_bytes = 0
        self.peak = self.measure_ffma_peak()

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def measure_ffma_peak(self):
        sink = torch.zeros(4, device=self.dev)
        flops = C.c_double(0)
        stream = torch.cuda.current_stream().cuda_stream
        peak = 0.0
        for _ in range(6):
            e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
            e0.record()
            self._lib.check(self.lib.ttrnn_ffma_probe(4000, sink.data_ptr(), C.byref(flops), stream), "ttrnn_ffma_probe")
            e1.record()
            torch.cuda.synchronize()
            peak = max(peak, flops.value / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        return peak

    def dump(self, out_dir, prefix, arrays):
        """Write each tensor as out_dir/<prefix><name>.npy (float32; float64 stays float64).  A tensor of more than
        DUMP_ELEMS elements is written as the flat elements at DUMP_ELEMS indices drawn from a generator seeded with 0,
        in ascending order: the same positions in every run, so two builds compare element for element."""
        os.makedirs(out_dir, exist_ok=True)
        for name, t in sorted(arrays.items()):
            t = t.detach()
            if t.numel() > DUMP_ELEMS:
                idx = torch.randint(t.numel(), (DUMP_ELEMS,), generator=torch.Generator().manual_seed(0)).sort().values
                a = t[torch.unravel_index(idx.to(t.device), t.shape)].cpu().numpy()
            else:
                a = t.cpu().numpy()
            if a.dtype != np.float64:
                a = a.astype(np.float32)
            self.dumped_bytes += a.nbytes
            if self.dumped_bytes > DUMP_BYTES:
                raise SystemExit("--dump-outputs: more than %d bytes of outputs" % DUMP_BYTES)
            np.save(os.path.join(out_dir, prefix + name + ".npy"), a)

    def run(self, cid, cfg, B_rank, steps, warmup, scaling, with_e2e=True, dump_dir=None):
        """One config at per-rank batch B_rank.  Returns the record (rank 0) or None.  With `dump_dir`, rank 0 writes
        what the last timed step computed there (see dump())."""
        from tensorized_rnn_b200.dist import allreduce_gradients
        lib, dev, dist = self.lib, self.dev, self.dist
        torch.manual_seed(cfg["seed"])
        dense = bool(cfg.get("dense"))
        ge2e = cfg.get("ge2e")
        if ge2e:
            with redirect_stdout(io.StringIO()):
                enc = self.tr.SpeakerEncoder(cfg["I"], cfg["H"], cfg["L"], ge2e[2], torch.device("cpu"), None, compression="tt",
                                             n_cores=cfg["d"], rank=cfg["r"]).to(dev)
            model = enc.rnn
        elif dense:
            model = (self.tr.LSTM if cfg["cell"] == "lstm" else self.tr.GRU)(cfg["I"], cfg["H"], cfg["L"], torch.device("cpu")).to(dev)
        else:
            cls = self.tr.TTLSTM if cfg["cell"] == "lstm" else self.tr.TTGRU
            with redirect_stdout(io.StringIO()):
                model = cls(cfg["I"], cfg["H"], cfg["L"], torch.device("cpu"), n_cores=cfg["d"], tt_rank=cfg["r"]).to(dev)
        named = list((enc if ge2e else model).named_parameters())
        params = [p for _, p in named]
        B, T, H = B_rank, cfg["T"], cfg["H"]
        if ge2e and B % ge2e[1] != 0:
            raise SystemExit("the GE2E step needs a per-rank batch that is a multiple of the utterances per speaker")
        c_rank = dict(cfg)
        c_rank["seed"] = cfg["seed"] + self.rank        # every rank owns different sequences
        x_host = make_input(c_rank, B).pin_memory()
        x_dev = x_host.to(dev)
        train = cfg["mode"] != "fwd"
        dense_dout = torch.rand(B, T, H, device=dev) if cfg["grad"] == "dense" else None

        def results(res):
            """What the recurrent stack returns to its caller: outputs and final state(s)."""
            if cfg["cell"] == "lstm":
                return {"out": res[0], "h_T": res[1][0], "c_T": res[1][1]}
            return {"out": res[0], "h_T": res[1]}

        def grads():
            return {"grad." + n: p.grad for n, p in named if p.grad is not None}

        def one_pass(x, keep=None):
            """One step; with a dict `keep`, also hands it what the step computed."""
            if not train:
                with torch.no_grad():
                    res = model(x)
                if keep is not None:
                    keep.update(results(res))
                return res[1][0] if cfg["cell"] == "lstm" else res[1]
            for p in params:
                p.grad = None
            if ge2e:
                embeds = enc(x)
                loss, _ = enc.loss(embeds.view(B // ge2e[1], ge2e[1], -1), group=(dist.group.WORLD if dist is not None else None))
                loss.backward()
                if dist is not None:
                    allreduce_gradients(params)
                if keep is not None:
                    keep.update(embeds=embeds, loss=loss, **grads())
                return loss
            res = model(x)
            if keep is not None:
                keep.update(results(res))
            out = res[0]
            hT = res[1][0] if cfg["cell"] == "lstm" else res[1]
            if dense_dout is not None:
                out.backward(dense_dout)
                result = hT
            else:
                loss = upstream(cfg, out, hT)
                loss.backward()
                result = loss
            if dist is not None:
                allreduce_gradients(params)             # one flat NCCL all-reduce of every TT-core / bias gradient
            if keep is not None:
                keep.update(grads())
            return result

        for _ in range(warmup):
            one_pass(x_dev)
        self.barrier()
        # ---- value: device-resident, per-step CUDA events, L2 flushed between steps -------------
        lib.ttrnn_launch_count(1)
        lib.ttrnn_tc_launch_count(1)

        def timed(n, keep=None):
            ev = []
            self.barrier()
            w0 = time.perf_counter()
            for i in range(n):
                self.flush_buf.fill_(1)
                e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
                e0.record()
                one_pass(x_dev, keep if i == n - 1 else None)
                e1.record()
                ev.append((e0, e1))
            self.barrier()
            self.windows.append((w0, time.perf_counter()))
            return sum(a.elapsed_time(b) for a, b in ev)

        last = {}
        total_ms = timed(steps, last)
        if dump_dir and self.rank == 0:
            self.dump(dump_dir, "cfg%d_" % cid, last)
        last.clear()
        launches = int(lib.ttrnn_launch_count(0))
        tc_launches = int(lib.ttrnn_tc_launch_count(0))
        # ---- per-kernel times: a second pass with the library's event pairs around every launch.  While that timing is
        # on, the library runs the row groups of a multi-layer stack back to back on one stream (per-launch events cannot
        # attribute time between kernels of two streams that share the SMs), so these are each kernel's OWN durations,
        # the figures an ncu launch list gives; `ms_per_step` above is the concurrent run.
        ksteps = min(steps, 5)
        lib.ttrnn_kernel_timing(1)
        serial_ms = timed(ksteps)
        lib.ttrnn_kernel_timing(0)
        nk = len(KINDS)
        kms = (C.c_double * nk)(*([0.0] * nk))
        kcnt = (C.c_int64 * nk)(*([0] * nk))
        lib.ttrnn_kernel_times(kms, kcnt)
        for i in range(nk):                            # scale to `steps` so that every consumer below divides by steps
            kms[i] = kms[i] * steps / ksteps
            kcnt[i] = int(kcnt[i] * steps / ksteps)
        # per-launch records of that pass: the recurrent kernels per variant (rows per CTA) and grid
        nrec = int(lib.ttrnn_kernel_launch_records(None, 0))
        rbuf = (C.c_double * (6 * max(nrec, 1)))()
        lib.ttrnn_kernel_launch_records(rbuf, nrec)
        variants = {}
        for i in range(nrec):
            kind, R, ctas, rows, tsteps, ms = (rbuf[6 * i + j] for j in range(6))
            if int(kind) not in (1, 2) or R <= 0:
                continue
            v = variants.setdefault((int(kind), int(R), int(ctas), int(rows)), {"launches": 0, "ms": 0.0, "row_steps": 0.0})
            v["launches"] += 1
            v["ms"] += ms
            v["row_steps"] += rows * tsteps

        # ---- e2e: pinned host input -> H2D -> module API -> D2H of the result, wall clock ----------
        e2e_ms, d2h = 0.0, 0
        if with_e2e:
            x_stage = torch.empty_like(x_dev)
            self.barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                x_stage.copy_(x_host, non_blocking=True)
                res = one_pass(x_stage)
                host = res.detach().to("cpu")           # D2H read of the step's result (loss / final state)
                d2h = host.numel() * host.element_size()
            self.barrier()
            e2e_ms = (time.perf_counter() - t0) * 1e3
            self.windows.append((t0, time.perf_counter()))
            del x_stage

        tot = torch.tensor([total_ms, e2e_ms], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(tot, op=dist.ReduceOp.MAX)
        total_ms, e2e_ms = float(tot[0]), float(tot[1])
        rec = None
        if self.rank == 0:
            world = self.world
            units = B * T * world * steps
            fwd_flops, hh_flops, ih_list, gate = algorithmic_flops(cfg)
            mult = 3 if train else 1
            if dense:
                plan = [{"path": "dense cells: batched tensor-core GEMMs + one step GEMM and one gate kernel per timestep"}]
                plan += [{"layer": l, "ih_route": "dense", "hh_dw": "dense_cell"} for l in range(cfg["L"])]
            else:
                plan = self._lib.describe_plan(model.spec().desc(B, T), training=train)
            layers = plan[1:]
            kern = {KINDS[i]: {"ms_per_step": kms[i] / steps, "launches_per_step": kcnt[i] / steps} for i in range(nk)}
            # algorithmic FLOPs credited to each kernel group per sequence-step (reference chain order; recomputed
            # forward work is NOT credited; where the hh core gradients are accumulated densely outside the recurrent
            # kernel the backward credit 2*F_hh is split half / half between k_rnn_bwd and gemm_dw)
            cred = {k: 0.0 for k in KINDS}
            for l, lay in enumerate(layers):
                route = lay.get("ih_route")
                ihf = ih_list[l]
                if route == "rank_one":
                    cred["k_rnn_fwd"] += ihf
                    if train:
                        cred["k_rnn_bwd"] += 2 * ihf
                elif route == "dense":
                    cred["gemm_ih_fwd"] += ihf
                    if train:
                        need_dx = l > 0
                        cred["gemm_dw"] += ihf
                        cred["gemm_dx" if need_dx else "gemm_dw"] += ihf
                else:
                    cred["k_ttlinear_fwd"] += ihf
                    if train:
                        cred["k_ttlinear_bwd"] += 2 * ihf
                if lay.get("hh_dw") == "dense_cell":
                    # dense cells: the step GEMMs are timed with the ih projection (gemm_ih_fwd / gemm_dx), gates in k_rnn_*
                    cred["gemm_ih_fwd"] += hh_flops
                    cred["k_rnn_fwd"] += gate
                    if train:
                        cred["gemm_dx"] += hh_flops
                        cred["gemm_dw"] += hh_flops
                        cred["k_rnn_bwd"] += 2 * gate
                    continue
                cred["k_rnn_fwd"] += hh_flops + gate
                if train:
                    if lay.get("hh_dw") == "dense":
                        cred["k_rnn_bwd"] += hh_flops + 2 * gate
                        cred["gemm_dw"] += hh_flops
                    elif lay.get("hh_dw") == "tt_chain":
                        cred["k_rnn_bwd"] += hh_flops + 2 * gate
                        cred["k_ttlinear_bwd"] += hh_flops
                    else:
                        cred["k_rnn_bwd"] += 2 * (hh_flops + gate)
            dom = max(range(nk), key=lambda i: kms[i])
            dom_ms = kms[dom] / steps
            achieved = cred[KINDS[dom]] * B * T / (dom_ms * 1e-3) / 1e12 if dom_ms > 0 else 0.0
            for i in range(nk):
                ms = kms[i] / steps
                kern[KINDS[i]]["credited_tflops"] = cred[KINDS[i]] * B * T / (ms * 1e-3) / 1e12 if ms > 0 else None
                kern[KINDS[i]]["frac_of_ffma_peak"] = (kern[KINDS[i]]["credited_tflops"] / self.peak
                                                       if ms > 0 and self.peak else None)
            # the recurrent kernels per variant: every (kind, rows per CTA, grid) is one template instantiation launched
            # with one grid; credited FLOPs of a launch = its rows x its timesteps x the per-layer credit of its kind
            sms = torch.cuda.get_device_properties(dev).multi_processor_count
            vlist = []
            for (kind, R, ctas, rows), v in sorted(variants.items()):
                per_layer = cred[KINDS[kind]] / cfg["L"]
                tf = per_layer * v["row_steps"] / (v["ms"] * 1e-3) / 1e12 if v["ms"] > 0 else 0.0
                vlist.append({"kernel": KINDS[kind], "rows_per_cta": R, "ctas": ctas, "rows": rows,
                              "launches_per_step": v["launches"] / ksteps, "ms_per_launch": v["ms"] / v["launches"],
                              "ms_per_step": v["ms"] / ksteps, "credited_tflops": tf,
                              "frac_of_ffma_peak": tf / self.peak if self.peak else None,
                              # the same on the SMs the grid occupies (one CTA per SM); the other SMs run the other row
                              # group's kernels in the concurrent run
                              "frac_on_occupied_sms": (tf / self.peak) * (sms / min(ctas, sms)) if self.peak and ctas else None})
            whole = mult * fwd_flops * B * T * steps / (total_ms * 1e-3) / 1e12
            # dominant KERNEL of the step = the instantiation (variant + grid) with the largest time per step; `achieved` =
            # its algorithmic FLOPs per launch / its average launch duration.  The aggregate over every variant of the same
            # kind (the round-1 definition) stays beside it as kind_group_frac.
            group_frac = achieved / self.peak if self.peak else None
            roof_kernel, flops_per_launch = KINDS[dom], None
            vd = max(vlist, key=lambda v: v["ms_per_step"]) if vlist else None
            if vd is not None and KINDS[dom] in ("k_rnn_fwd", "k_rnn_bwd") and vd["kernel"] == KINDS[dom]:
                roof_kernel = "%s (%d rows per CTA, %d CTAs, %d rows per launch)" % (vd["kernel"], vd["rows_per_cta"], vd["ctas"], vd["rows"])
                achieved = vd["credited_tflops"]
                flops_per_launch = vd["credited_tflops"] * 1e12 * vd["ms_per_launch"] * 1e-3
            traffic = None
            try:
                with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                    ent = json.load(f).get(cfg["name"].split(" ")[0])
                if ent and ent["kernel"] == KINDS[dom]:
                    traffic = ent["dram_bytes_per_launch"]
            except Exception:
                traffic = None
            rec = {
                "config_id": cid, "config": config_json(cfg, B, world, scaling), "scaling": scaling,
                "value": units / (total_ms * 1e-3), "unit": "cell-steps/s",
                "layer_cell_steps_per_s": units * cfg["L"] / (total_ms * 1e-3),
                "ms_per_step": total_ms / steps, "steps": steps, "warmup": warmup,
                "ms_per_step_kernel_timing_pass": serial_ms / ksteps,
                "e2e": ({"value": units / (e2e_ms * 1e-3), "unit": "cell-steps/s", "h2d_bytes_per_step": x_host.numel() * 4,
                         "d2h_bytes_per_step": d2h} if with_e2e else None),
                "gpu_launches": launches, "tc_gemm_launches": tc_launches,
                "roofline": {"bound": "fp32_ffma", "kernel": roof_kernel, "achieved": achieved, "peak": self.peak,
                             "unit": "TFLOP/s", "frac": achieved / self.peak if self.peak else None, "traffic": traffic,
                             "algorithmic_flops_per_launch": flops_per_launch,
                             "kind_group": KINDS[dom], "kind_group_frac": group_frac,
                             "traffic_unit": "bytes per launch (ncu dram read+write, profiles/)",
                             "peak_source": "ttrnn_ffma_probe measured in this run (MEASURED_PEAKS.json has no FP32 entry)",
                             "algorithmic_flops_per_seqstep": cred[KINDS[dom]],
                             "whole_step_tflops_per_gpu": whole, "whole_step_frac": whole / self.peak if self.peak else None,
                             "fwd_flops_per_seqstep": fwd_flops, "kernels": kern, "recurrent_variants": vlist,
                             "kernel_times": "second pass of %d steps with an event pair around every launch; row groups run "
                                             "back to back in that pass, so these are each kernel's own durations (what an ncu "
                                             "launch list gives), while ms_per_step is the concurrent run" % ksteps,
                             "plan": plan,
                             # the second bound SURVEY.md 8d asks for: the sequential chain.  A CTA owns its rows for all T, so a
                             # layer-pass cannot be shorter than T x (per-step dependency chain); these are the measured per-step
                             # times of the recurrent kernels (all row tiles of a layer run concurrently when they fit the SMs)
                             "recurrent_us_per_layer_step": {
                                 "fwd": kms[1] / steps / (cfg["L"] * T) * 1e3, "bwd": kms[2] / steps / (cfg["L"] * T) * 1e3}},
            }
        del model, params, x_dev, x_host, dense_dout
        torch.cuda.empty_cache()
        return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps of every config (default: 10; 5 for cfg4, 3 for cfg5)")
    ap.add_argument("--warmup", type=int, default=None, help="untimed warm-up steps of every config (default: 3)")
    ap.add_argument("--headline", type=int, default=3, choices=sorted(CONFIGS))
    ap.add_argument("--config", type=int, default=0, help="shorthand: headline = this config and run only it")
    ap.add_argument("--configs", default="1,2,3,4,5,6,7,8,9", help="configs measured into all_configs")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="override the global batch of the headline config (profiling)")
    ap.add_argument("--seq-len", type=int, default=0, help="override T of the headline config (profiling only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-weak", action="store_true", help="N > 1: skip the weak-scaling measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of every config computed (outputs, final states, parameter "
                         "gradients) as DIR/cfg<id>_<name>.npy")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup is not None and args.warmup < 0:
        ap.error("--warmup must not be negative")

    def steps_for(cid):
        dw, ds = STEP_DEFAULT.get(cid, (3, 10))
        return (dw if args.warmup is None else args.warmup), (ds if args.steps is None else args.steps)

    if args.config:
        args.headline, args.configs = args.config, str(args.config)
    ids = [int(v) for v in args.configs.split(",") if v.strip()]
    if args.headline not in ids:
        ids.append(args.headline)
    cfgs = {i: dict(CONFIGS[i]) for i in ids}
    head = cfgs[args.headline]
    if args.batch:
        head["B"] = args.batch
    if args.seq_len:
        head["T"] = args.seq_len
        head["name"] += " [T overridden to %d: profiling run]" % args.seq_len
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    metric = "TT-%s cell-steps/sec (batch x T), %s" % ("LSTM" if head["cell"] == "lstm" else "GRU", head["mode"])

    # ---------------- reference arm: the CPU path on the host cores --------------------------
    if args.impl == "reference":
        if rank != 0:
            return 0
        # batch of the bounded sample: a pilot pass at batch 32 sizes it so that (warmup + steps) passes take ~150 s;
        # T stays at the config value (the reference's cost is per-step dispatch and its O(T^2) backward)
        T = head["T"]
        warmup, steps = steps_for(args.headline)
        _, pilot = run_cpu_oracle(head, 32, T, 1, 0)
        budget = 150.0 / (steps + warmup)
        Bs = int(max(16, min(head["B"], 32 * budget / pilot)))
        Bs = max(16, (Bs // 16) * 16) if Bs < head["B"] else head["B"]
        val, sec = run_cpu_oracle(head, Bs, T, steps, warmup)
        sample = "batch %d of the config's %d sequences x T %d per step (pilot pass at batch 32 took %.1f s); oracle port of " \
                 "the reference PyTorch path, %d threads" % (Bs, head["B"], T, pilot, torch.get_num_threads())
        cj = config_json(head, Bs, 1, "none")
        cj["parallelism"] = "host CPU, %d threads" % torch.get_num_threads()
        cj["sample_of_global_batch"] = head["B"]
        line = {"impl": "reference", "metric": metric, "value": val, "unit": "cell-steps/s", "n_gpus": args.gpus,
                "steps": steps, "warmup": warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cj,
                "sample": sample,
                "cpu_baseline": {"value": val, "unit": "cell-steps/s", "cores": torch.get_num_threads(), "kind": "port",
                                 "sample": sample, "batch": Bs, "seq_len": T},
                "e2e": {"value": val, "unit": "cell-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    # ---------------- our arm -----------------------------------------------------------------
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path")
    # stdout carries exactly ONE line (the JSON record): anything libraries print while we run (NCCL prints its version
    # banner to stdout at the first collective) is diverted to stderr at the file-descriptor level
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    gb = GpuBench(rank, world, local_rank)

    def split(B):
        return (B + world - 1) // world

    records = []
    head_rec = None
    order = [args.headline] + [i for i in ids if i != args.headline]
    if world > 1:
        # the dense baseline is a single-GPU comparison line (dense vs TT on one device path); its per-step GEMMs fall back to
        # FFMA below 128 rows per GPU, which says nothing about the TT path that is being scaled
        order = [i for i in order if not cfgs[i].get("dense") or i == args.headline]
    for cid in order:
        cfg = cfgs[cid]
        w, s = steps_for(cid)
        rec = gb.run(cid, cfg, split(cfg["B"]), s, w, "strong", dump_dir=args.dump_outputs)
        weak = None
        if world > 1 and not args.no_weak:
            weak = gb.run(cid, cfg, cfg["B"], min(s, 5), min(w, 3), "weak", with_e2e=False)
        if rank == 0:
            if weak is not None:
                rec["weak"] = {"value": weak["value"], "ms_per_step": weak["ms_per_step"], "batch_per_gpu": cfg["B"],
                               "global_batch": cfg["B"] * world}
            records.append(rec)
            if cid == args.headline:
                head_rec = rec

    if rank == 0:
        sampler.stop()
        clocks = sampler.summary(gb.windows)
        # CPU baseline (N = 1 only): bounded sample per config, batch stated
        if world == 1 and not args.no_cpu_baseline:
            for rec in records:
                cid = rec["config_id"]
                Bs, Ts = CPU_SAMPLE[cid]
                Ts = min(Ts, cfgs[cid]["T"])
                val, sec = run_cpu_oracle(cfgs[cid], Bs, Ts, 1, 0)
                rec["cpu_baseline"] = {"value": val, "unit": "cell-steps/s", "cores": torch.get_num_threads(), "kind": "port",
                                       "seconds": sec, "batch": Bs, "seq_len": Ts,
                                       "sample": "batch %d x T %d of the workload (global batch %d, T %d), 1 pass, oracle port "
                                                 "of the reference PyTorch path" % (Bs, Ts, cfgs[cid]["B"], cfgs[cid]["T"])}
        line = {
            "metric": metric, "value": head_rec["value"], "unit": "cell-steps/s", "n_gpus": world,
            "steps": head_rec["steps"], "warmup": head_rec["warmup"], "ms_per_step": head_rec["ms_per_step"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic (random-init TT cores, %s input)" % head["inp"],
            "config": head_rec["config"], "e2e": head_rec["e2e"], "gpu_launches": head_rec["gpu_launches"],
            "clocks": clocks, "roofline": head_rec["roofline"],
        }
        if "weak" in head_rec:
            line["weak"] = head_rec["weak"]
        if "cpu_baseline" in head_rec:
            line["cpu_baseline"] = head_rec["cpu_baseline"]
        line["all_configs"] = [{k: v for k, v in r.items() if k != "config_id"} | {"id": r["config_id"]} for r in records]
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line))
        sys.stdout.flush()
        os.dup2(2, 1)
    if gb.dist is not None:
        gb.dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
