"""Cost of a learned-variance model (UbConfig.learn_sigma, guided-diffusion's `--learn_sigma True`) against the plain
model.

    python tools/learn_sigma_bench.py [--rounds 5] [--steps 50] [--B 32] [--out FILE]

Two trainers of the default 64x64 model at batch B, learn_sigma = 1 and learn_sigma = 0, perturb_zero_params weights,
one device-resident batch (x0 ~ U[-1, 1]).  Every round times both arms, alternating:
  step_ms       `steps` captured training steps (ub_trainer_train_step_device), CUDA events around the loop
  ddim50_ms     one ub_trainer_sample_spaced call over space_timesteps(1000, "ddim50"), host clock (the call synchronises)
  ancestral250_ms  one learned-range (plain arm: fixed-large) ancestral call over space_timesteps(1000, "250")
Then one ub_trainer_profile per arm (CUDA events around every launch, 3 repetitions) gives the UB_KIND_SMALL class (the
3-channel convs, the embedding MLPs, the output conv with the loss) and the output head's forward and backward launches
from the per-op dump.  The median over the rounds is reported with the spread (min .. max).  The card name, power limit
and maximum SM clock are read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
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


def profile_ops(tr):
    """ub_trainer_profile plus its per-op dump: (class times, {label: us})."""
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "ops.tsv")
        os.environ["UB_PROFILE_DUMP"] = path
        try:
            prof = tr.profile(3)
        finally:
            del os.environ["UB_PROFILE_DUMP"]
        ops = {}
        with open(path) as fh:
            for line in fh:
                cols = line.rstrip("\n").split("\t")
                if len(cols) >= 7 and cols[6]:
                    ops[cols[6]] = float(cols[3])
    return prof, ops


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--B", type=int, default=32)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("learn_sigma_bench needs a CUDA device")
    import unet_oracle as O
    ub = ge.load_package()
    g = torch.Generator().manual_seed(0)
    x0 = (torch.rand(a.B, 3, 64, 64, generator=g) * 2 - 1).cuda()
    calls = {"ddim50_ms": (ub.space_timesteps(1000, "ddim50"), "ddim"),
             "ancestral250_ms": (ub.space_timesteps(1000, "250"), "ancestral")}
    arms = {}
    for name, ls in (("learn_sigma", 1), ("plain", 0)):
        cfg = O.UNetConfig(out_channels=6 if ls else 3)
        flat = O.perturb_zero_params(cfg, O.flatten_params(cfg, O.init_params(cfg, seed=0)))
        tr = ub.Trainer(B=a.B, learn_sigma=ls)
        tr.set_params(flat.numpy())
        arms[name] = tr
        for _ in range(5):  # warm-up: graph capture, module load
            tr.train_step_device(x0.data_ptr())
        tr.sync()
        tr.sample_spaced(None, calls["ddim50_ms"][0], "ddim", 0.0, True, None, 1)
    res = {n: {"step_ms": [], **{k: [] for k in calls}} for n in arms}
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
            res[name]["step_ms"].append(ev0.elapsed_time(ev1) / a.steps)
            for k, (ts, sampler) in calls.items():
                t0 = time.perf_counter()
                tr.sample_spaced(None, ts, sampler, 0.0, True, None, 2)
                res[name][k].append((time.perf_counter() - t0) * 1e3)
    out = {"card": card(), "B": a.B, "steps": a.steps, "rounds": a.rounds}
    for name, tr in arms.items():
        r = {k: {"median": statistics.median(v), "min": min(v), "max": max(v)} for k, v in res[name].items()}
        prof, ops = profile_ops(tr)
        r["small_class_ms"] = prof["small"]["ms"]
        r["profile_total_ms"] = prof["total_ms"]
        r["launches_per_step"] = tr.launches_per_step()
        r["ops_us"] = {k: v for k, v in ops.items() if k.startswith("output conv")}
        out[name] = r
        tr.close()
    s, p = out["learn_sigma"], out["plain"]
    out["delta"] = {"step_ms": s["step_ms"]["median"] - p["step_ms"]["median"],
                    "small_class_ms": s["small_class_ms"] - p["small_class_ms"],
                    **{k: s[k]["median"] - p[k]["median"] for k in calls}}
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    np.set_printoptions(precision=4)
    main()
