"""Cost of classifier-free guidance (UbConfig.class_dropout, ub_trainer_set_guidance).

    python tools/cfg_bench.py [--rounds 5] [--steps 50] [--B 32] [--out FILE]

Training: two trainers of the default 64x64 model at batch B with num_classes = 10, one with class_dropout = 0.1 (the
label-drop kernel in the captured step, an 11th label row), perturb_zero_params weights of the matching oracle model,
one device-resident batch (x0 ~ U[-1, 1]), labels 0..9 repeated.  `steps` captured training steps
(ub_trainer_train_step_device), CUDA events around the loop.
Sampling: the class_dropout trainer, one ub_trainer_sample_spaced call over space_timesteps(1000, "ddim50") at
guidance scale 1 (one forward per iteration) and at scale 3 (two), host clock (the call synchronises).
Every round times all four, alternating the arms; the median over the rounds is reported with the spread
(min .. max).  The card name, power limit and maximum SM clock are read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import __graft_entry__ as ge  # noqa: E402


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60)
        if r.returncode == 0 and r.stdout.strip():
            return r.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pass
    return torch.cuda.get_device_name() + ", power limit not readable"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--B", type=int, default=32)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("cfg_bench needs a CUDA device")
    import unet_oracle as O
    ub = ge.load_package()
    g = torch.Generator().manual_seed(0)
    x0 = (torch.rand(a.B, 3, 64, 64, generator=g) * 2 - 1).cuda()
    labels = (np.arange(a.B) % 10).astype(np.int32)
    ts = ub.space_timesteps(1000, "ddim50")
    arms = {}
    for name, p in (("class_conditional", 0.0), ("class_dropout_0.1", 0.1)):
        cfg = O.UNetConfig(num_classes=10 + (1 if p else 0))
        flat = O.perturb_zero_params(cfg, O.flatten_params(cfg, O.init_params(cfg, seed=0)))
        tr = ub.Trainer(B=a.B, num_classes=10, class_dropout=p)
        tr.set_params(flat.numpy())
        tr.set_labels(labels)
        arms[name] = tr
        for _ in range(5):  # warm-up: graph capture, module load
            tr.train_step_device(x0.data_ptr())
        tr.sync()
    guided = arms["class_dropout_0.1"]
    for s in (1.0, 3.0):  # warm-up of both sampling graphs
        guided.set_guidance(s)
        guided.sample_spaced(None, ts, "ddim", 0.0, True, None, 1)
    step = {n: [] for n in arms}
    ddim = {1.0: [], 3.0: []}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(a.rounds):
        for name, tr in arms.items():
            st = torch.cuda.ExternalStream(tr.stream())
            tr.sync()
            ev0.record(st)
            for _ in range(a.steps):
                tr.train_step_device(x0.data_ptr())
            ev1.record(st)
            ev1.synchronize()
            step[name].append(ev0.elapsed_time(ev1) / a.steps)
        for s in (1.0, 3.0):
            guided.set_guidance(s)
            t0 = time.perf_counter()
            guided.sample_spaced(None, ts, "ddim", 0.0, True, None, 2)
            ddim[s].append((time.perf_counter() - t0) * 1e3)
    stat = lambda v: {"median": statistics.median(v), "min": min(v), "max": max(v)}
    out = {"card": card(), "B": a.B, "steps": a.steps, "rounds": a.rounds,
           "train_step_ms": {n: stat(v) for n, v in step.items()},
           "launches_per_step": {n: tr.launches_per_step() for n, tr in arms.items()},
           "ddim50_ms": {f"scale_{s:g}": stat(v) for s, v in ddim.items()}}
    out["delta"] = {
        "train_step_ms": out["train_step_ms"]["class_dropout_0.1"]["median"]
        - out["train_step_ms"]["class_conditional"]["median"],
        "ddim50_ratio_scale3_over_scale1": out["ddim50_ms"]["scale_3"]["median"] / out["ddim50_ms"]["scale_1"]["median"]}
    for tr in arms.values():
        tr.close()
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
