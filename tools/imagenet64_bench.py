"""Step and sampling time of guided-diffusion's ImageNet 64x64 model, linear against cosine noise schedule.

    python tools/imagenet64_bench.py [--rounds 5] [--steps 10] [--B 32] [--out FILE]

The model of guided-diffusion's `--attention_resolutions 32,16,8 --class_cond True --learn_sigma True --num_channels 192
--num_head_channels 64 --num_res_blocks 3 --resblock_updown True --use_scale_shift_norm True --dropout 0.1`
(295 904 454 parameters) with noise_schedule = linear and cosine: two trainers at batch B (halved until one is created,
the batch used is reported), perturb_zero_params weights, one device-resident batch (x0 ~ U[-1, 1]), labels 0..B-1.
Every round times both arms, alternating:
  step_ms    `steps` captured training steps (ub_trainer_train_step_device), CUDA events around the loop
  ddim50_ms  one ub_trainer_sample_spaced call over space_timesteps(1000, "ddim50"), host clock (the call synchronises)
Then one ub_trainer_profile per arm (CUDA events around every launch, 3 repetitions) splits a step by kernel class.
The schedule only changes table contents, so the arms should agree.  The median over the rounds is reported with the
spread (min .. max).  The card name, power limit and maximum SM clock are read in the same run."""
import argparse
import json
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import __graft_entry__ as ge  # noqa: E402
from learn_sigma_bench import card  # noqa: E402

IMAGENET64 = dict(att_start_level=1, num_classes=1000, learn_sigma=1, C_model=192, head_size=64, n_res_blocks=3,
                  resblock_updown=1, use_scale_shift_norm=1, dropout=0.1)
ORACLE = dict(attn_start_level=1, num_classes=1000, out_channels=6, model_channels=192, head_size=64, num_res_blocks=3,
              resblock_updown=True, use_scale_shift_norm=True, dropout=0.1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--B", type=int, default=32)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("imagenet64_bench needs a CUDA device")
    import numpy as np
    import unet_oracle as O
    ub = ge.load_package()
    cfg = O.UNetConfig(**ORACLE)
    flat = O.perturb_zero_params(cfg, O.flatten_params(cfg, O.init_params(cfg, seed=0))).numpy()
    B, arms = a.B, {}
    while not arms:
        try:
            for name, s in (("linear", 0), ("cosine", 1)):
                arms[name] = ub.Trainer(B=B, noise_schedule=s, **IMAGENET64)
        except ub.UbError as e:  # out of memory: try half the batch
            print(f"B = {B}: {e}", file=sys.stderr)
            for tr in arms.values():
                tr.close()
            arms, B = {}, B // 2
            if B < 1:
                raise
    g = torch.Generator().manual_seed(0)
    x0 = (torch.rand(B, 3, 64, 64, generator=g) * 2 - 1).cuda()
    ddim50 = ub.space_timesteps(1000, "ddim50")
    for tr in arms.values():
        tr.set_params(flat)
        tr.set_labels(np.arange(B, dtype=np.int32))
        for _ in range(3):  # warm-up: graph capture, module load
            tr.train_step_device(x0.data_ptr())
        tr.sync()
        tr.sample_spaced(None, ddim50, "ddim", 0.0, True, None, 1)
    res = {n: {"step_ms": [], "ddim50_ms": []} for n in arms}
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
            t0 = time.perf_counter()
            tr.sample_spaced(None, ddim50, "ddim", 0.0, True, None, 2)
            res[name]["ddim50_ms"].append((time.perf_counter() - t0) * 1e3)
    out = {"card": card(), "B": B, "B_requested": a.B, "steps": a.steps, "rounds": a.rounds,
           "nparams": arms["linear"].nparams}
    for name, tr in arms.items():
        r = {k: {"median": statistics.median(v), "min": min(v), "max": max(v)} for k, v in res[name].items()}
        prof = tr.profile(3)
        r["profile_ms"] = {k: round(v["ms"], 4) for k, v in prof.items() if k != "total_ms"}
        r["profile_launches"] = {k: v["launches"] for k, v in prof.items() if k != "total_ms"}
        r["profile_total_ms"] = prof["total_ms"]
        r["images_per_s"] = B / (r["step_ms"]["median"] / 1e3)
        out[name] = r
        tr.close()
    out["cosine_over_linear"] = {k: out["cosine"][k]["median"] / out["linear"][k]["median"]
                                 for k in ("step_ms", "ddim50_ms")}
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
