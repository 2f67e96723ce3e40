"""Attention core at head size 32 vs 64 on the trainer's shapes, and the default training step at both head sizes.

    python tools/attn_bench.py [--reps 200] [--rounds 5] [--steps 20] [--out FILE]

Kernels: the tcgen05 attention core (ub_attention_nhwc_forward / _backward, impl 0) for the attention levels of the
default 64x64 model at B = 32 (T = 256 with C = 192, T = 64 with C = 256) and of the 128x128 five-level model at B = 64
(same T and C).  For each shape and head size a CUDA graph of `reps` forward (or backward) calls is captured and
replayed `rounds` times; the time per call is CUDA-event time over the replay divided by `reps`, head size 32 and 64
alternating round by round.  The graph keeps the host's per-call planning (tensor-map encoding) out of the device
timeline.  Inputs stay resident in L2 (a few MB), as in the trainer, where the qkv conv has just written them.  The
backward here runs its dq and dkv kernels one after the other on one stream; the trainer runs them side by side.
FLOP counts: forward 4*B*T^2*C, backward 10*B*T^2*C (the trainer's profile counts), the same for both head sizes.

Training step: the default model (64x64, B = 32, captured-graph train_step on a device batch) at head_size 32 and 64,
alternating in `rounds` rounds of `steps` steps, CUDA events on the trainer's stream.

The card name and power limit are read in the same run and printed with the numbers."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import __graft_entry__ as ge  # noqa: E402

SHAPES = [  # (what, B, T, C)
    ("default 64x64, 16x16 level", 32, 256, 192),
    ("default 64x64, 8x8 level", 32, 64, 256),
    ("config 5 128x128, 16x16 level", 64, 256, 192),
    ("config 5 128x128, 8x8 level", 64, 64, 256),
]


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60)
        if r.returncode == 0 and r.stdout.strip():
            return r.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pass
    return torch.cuda.get_device_name() + ", power limit not readable"


class AttnCase:
    def __init__(self, L, B, T, Cc, hs):
        self.L, self.B, self.T, self.C, self.NH = L, B, T, Cc, Cc // hs
        g = torch.Generator(device="cuda").manual_seed(3)
        bf = dict(dtype=torch.bfloat16, device="cuda")
        self.qkv = (torch.randn(B * T, 3 * Cc, generator=g, device="cuda") * 1.5).to(torch.bfloat16)
        self.dout = torch.randn(B * T, Cc, generator=g, device="cuda").to(torch.bfloat16)
        self.out = torch.empty(B * T, Cc, **bf)
        self.dqkv = torch.empty(B * T, 3 * Cc, **bf)
        self.lse = torch.empty(B, self.NH, T, dtype=torch.float32, device="cuda")
        self.dsum = torch.empty_like(self.lse)

    def fwd(self):
        p = lambda t: C.c_void_p(t.data_ptr())
        rc = self.L.ub_attention_nhwc_forward(p(self.qkv), p(self.out), p(self.lse), self.B, self.T, self.C, self.NH, 0)
        assert rc == 0, self.L.ub_last_error()

    def bwd(self):
        p = lambda t: C.c_void_p(t.data_ptr())
        rc = self.L.ub_attention_nhwc_backward(p(self.qkv), p(self.out), p(self.dout), p(self.lse), p(self.dqkv),
                                               p(self.dsum), self.B, self.T, self.C, self.NH, 0)
        assert rc == 0, self.L.ub_last_error()

    def graph(self, fn, reps):
        """CUDA graph of `reps` calls of fn; the layer operators are pointed at the capture stream meanwhile."""
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self.L.ub_set_stream(C.c_void_p(s.cuda_stream))
            for _ in range(3):
                fn()  # warm-up: module load, smem attributes
            s.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                self.L.ub_set_stream(C.c_void_p(s.cuda_stream))
                for _ in range(reps):
                    fn()
            self.L.ub_set_stream(None)
        torch.cuda.synchronize()
        return g


def time_graph(g, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / reps  # us per call


def bench_kernels(ub, reps, rounds, log):
    L = ub.lib()
    rows = []
    for what, B, T, Cc in SHAPES:
        cases = {hs: AttnCase(L, B, T, Cc, hs) for hs in (32, 64)}
        graphs = {(hs, d): cases[hs].graph(cases[hs].fwd if d == "fwd" else cases[hs].bwd, reps)
                  for hs in (32, 64) for d in ("fwd", "bwd")}
        for g in graphs.values():
            g.replay()  # warm replay
        torch.cuda.synchronize()
        times = {k: [] for k in graphs}
        for _ in range(rounds):
            for d in ("fwd", "bwd"):
                for hs in (32, 64):
                    times[(hs, d)].append(time_graph(graphs[(hs, d)], reps))
        for d in ("fwd", "bwd"):
            flop = (4.0 if d == "fwd" else 10.0) * B * T * T * Cc
            for hs in (32, 64):
                ts = times[(hs, d)]
                med = statistics.median(ts)
                r = dict(kind="attn", shape=what, B=B, T=T, C=Cc, head_size=hs, NH=Cc // hs, dir=d, us_median=med,
                         us_min=min(ts), us_max=max(ts), tflops=flop / med * 1e-6)
                rows.append(r)
                log(json.dumps(r))
            r32 = statistics.median(times[(32, d)])
            r64 = statistics.median(times[(64, d)])
            log(f"# {what:32s} B={B:3d} T={T:3d} C={Cc:3d} {d}: hs32 {r32:8.1f} us  hs64 {r64:8.1f} us  "
                f"(hs64/hs32 {r64 / r32:.3f})")
        del graphs, cases
        torch.cuda.synchronize()
    return rows


def bench_steps(ub, steps, rounds, log):
    import unet_oracle as O
    B = 32
    flat = O.flatten_params(O.UNetConfig(), O.init_params(O.UNetConfig(), seed=0)).numpy()
    trs = {hs: ub.Trainer(B=B, head_size=hs) for hs in (32, 64)}
    x = (torch.rand(B, 3, 64, 64, generator=torch.Generator().manual_seed(7)) * 2 - 1).cuda()
    for tr in trs.values():
        tr.set_params(flat)
        for _ in range(5):
            tr.train_step_device(x.data_ptr())
        tr.sync()
    ms = {hs: [] for hs in trs}
    for _ in range(rounds):
        for hs, tr in trs.items():
            st = torch.cuda.ExternalStream(tr.stream())
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record(st)
            for _ in range(steps):
                tr.train_step_device(x.data_ptr())
            e1.record(st)
            tr.sync()
            ms[hs].append(e0.elapsed_time(e1) / steps)
    rows = []
    for hs in trs:
        r = dict(kind="train_step", model="default 64x64", B=B, head_size=hs, steps_per_round=steps,
                 ms_per_step_median=statistics.median(ms[hs]), ms_per_step_rounds=ms[hs],
                 last_loss=trs[hs].last_loss())
        rows.append(r)
        log(json.dumps(r))
    log(f"# default training step B=32: hs32 {statistics.median(ms[32]):.3f} ms  hs64 {statistics.median(ms[64]):.3f} ms")
    for tr in trs.values():
        tr.close()
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=200, help="calls per captured graph")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20, help="training steps per round")
    ap.add_argument("--no-steps", action="store_true", help="kernels only")
    ap.add_argument("--out", default=None, help="also write the log to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("attn_bench: no CUDA device")
    ub = ge.load_package()
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log(f"# card: {card()}")
    log(f"# tcgen05 attention core, CUDA graphs of {a.reps} calls, {a.rounds} rounds alternating head size; "
        f"us per call, median (min/max in the JSON)")
    bench_kernels(ub, a.reps, a.rounds, log)
    if not a.no_steps:
        bench_steps(ub, a.steps, a.rounds, log)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
