"""Sampling time of the trainer: generate.py's full DDPM loop against guided-diffusion's respaced samplers.

    python tools/sample_bench.py [--rounds 3] [--B 32] [--out FILE]

The default 64x64 model at B = 32 with perturb_zero_params weights (the zero-initialised layers perturbed, so that
every layer carries signal).  Modes, one batch of B images each, x_T drawn on the device:
  generate     ub_trainer_sample over its full range t = 999 .. 2 (998 iterations)
  ddim50       ub_trainer_sample_spaced, DDIM eta = 0 over space_timesteps(1000, "ddim50")
  ddim250      the same over "ddim250"
  ancestral250 ub_trainer_sample_spaced, ancestral over "250"
Every mode runs once as warm-up (graph capture, module load), then the modes alternate in `rounds` rounds.  A batch
is timed with the host clock around the call, which ends in a stream synchronise; it includes the call's host work and
its copies (x_T is drawn on the device, the B images come back).  ms/iteration is that time over the number of U-Net
forwards; images/s is B over the batch time.  The median over the rounds is reported, with the spread (min .. max).

The card name, power limit and maximum SM clock are read in the same run and printed with the numbers."""
import argparse
import os
import statistics
import subprocess
import sys
import time

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
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--B", type=int, default=32)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("sample_bench needs a CUDA device")
    import unet_oracle as O
    ub = ge.load_package()
    cfg = O.UNetConfig()
    flat = O.perturb_zero_params(cfg, O.flatten_params(cfg, O.init_params(cfg, seed=0)))
    tr = ub.Trainer(B=a.B)
    tr.set_params(flat.numpy())
    modes = {
        "generate": (998, lambda s: tr.sample(None, -1, -1, None, seed=s)),
        "ddim50": (50, lambda s: tr.sample_spaced(None, ub.space_timesteps(1000, "ddim50"), "ddim", 0.0, True, None, s)),
        "ddim250": (250, lambda s: tr.sample_spaced(None, ub.space_timesteps(1000, "ddim250"), "ddim", 0.0, True, None,
                                                    s)),
        "ancestral250": (250, lambda s: tr.sample_spaced(None, ub.space_timesteps(1000, "250"), "ancestral", 0.0, True,
                                                         None, s)),
    }
    for _, fn in modes.values():  # warm-up
        fn(0)
    times = {k: [] for k in modes}
    for r in range(a.rounds):
        for k, (_, fn) in modes.items():
            t0 = time.perf_counter()
            x = fn(r + 1)
            times[k].append(time.perf_counter() - t0)
            assert x.shape == (a.B, 3, 64, 64) and bool(torch.isfinite(torch.from_numpy(x)).all()), k
    tr.close()
    lines = [f"# tools/sample_bench.py --rounds {a.rounds} --B {a.B}",
             f"# card: {card()}",
             f"# default 64x64 model, B = {a.B}, perturb_zero_params weights; median over {a.rounds} alternating rounds "
             "after one warm-up batch per mode",
             f"{'mode':<14}{'iterations':>11}{'ms/iteration':>14}{'s/batch':>10}{'images/s':>10}{'vs generate':>13}"
             "   s/batch min .. max"]
    base = statistics.median(times["generate"])
    for k, (n, _) in modes.items():
        s = statistics.median(times[k])
        lines.append(f"{k:<14}{n:>11}{1e3 * s / n:>14.3f}{s:>10.3f}{a.B / s:>10.1f}{base / s:>12.1f}x   "
                     f"{min(times[k]):.3f} .. {max(times[k]):.3f}")
    text = "\n".join(lines) + "\n"
    print(text, end="")
    if a.out:
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
