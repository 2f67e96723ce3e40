#!/usr/bin/env python
"""bench.py -- UNet-64 diffusion training step throughput (BASELINE.json metric) on N B200s.

    python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
    python bench.py --impl reference --gpus N ...          # the reference's CPU (PyTorch) path, oracle port
    python bench.py ... --dump-outputs DIR                 # also write the last timed step's outputs as DIR/*.npy

One "step" = the loop body of train_unet.cu:5019-5037 on one synthetic batch: H2D batch copy (e2e only),
timestep + noise draw, q-sample, U-Net forward, MSE, backward, (gradient all-reduce), AdamW.
Workload at N=1: BASELINE.json configs[2] -- default 64x64 unconditional U-Net (20 494 211 params), batch 32.
N>1: weak scaling, batch 32 per GPU (N=8 is configs[3]: global batch 256), gradients all-reduced over NCCL.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "UNet-64 train images/sec"
UNIT = "images/s"
FLOP_PER_IMG_FWD_BWD = 38.76e9  # BASELINE.md section 3 (tensor FLOPs, fwd + bwd)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])), mx.append(float(c[2]))
            except ValueError:
                continue
            for n, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


# ---------------------------------------------------------------------------------------------------- CPU arm
def cpu_step_timer(B: int, steps: int, warmup: int):
    """Time the oracle port (the reference's PyTorch-CPU path restated, oracle/unet_oracle.py) on all host cores."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import unet_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = O.UNetConfig()
    flat = O.flatten_params(cfg, O.init_params(cfg, seed=0))
    m, v = torch.zeros_like(flat), torch.zeros_like(flat)
    times = []
    for i in range(warmup + steps):
        x0, t, noise = O.synthetic_batch(cfg, B, seed=1234 + i)
        t0 = time.perf_counter()
        _, _, g = O.train_step_grads(cfg, flat, x0, t, noise)
        flat, m, v = O.adamw_step(flat, g, m, v, i + 1, lr=1e-4)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return sum(times) / len(times), cores, torch.get_num_threads()


def cpu_sample_batch(budget_s: float, n_steps: int) -> int:
    """Largest batch in {32, 16, 8, 4} whose n_steps CPU steps fit the time budget (probe: one batch-4 step)."""
    sec4, _, _ = cpu_step_timer(4, 1, 0)
    for B in (32, 16, 8):
        if sec4 * (B / 4.0) * n_steps <= budget_s:   # the CPU path scales ~linearly with the batch
            return B
    return 4


def run_reference(args):
    """The reference's own CPU implementation of the path (its PyTorch ground truth, restated in oracle/unet_oracle.py and
    pinned against it) on all host cores, on this arm's config: default 64x64 U-Net, full train step, batch 32 per step
    unless that would not finish within a few minutes on this box (then a smaller, stated, sample of the batch)."""
    rank, _, world = dist_env()
    if rank != 0:
        return
    n = args.steps + args.warmup
    B = cpu_sample_batch(240.0, n)
    sec, cores, threads = cpu_step_timer(B, args.steps, args.warmup)
    val = B / sec
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "train_unet default 64x64 unconditional U-Net (20494211 params, channel_mult 1-2-3-4, "
                               "attention at 16x16 and 8x8), full train step (q-sample, fwd, MSE, bwd, AdamW)",
                   "batch_per_gpu": 32, "global_batch": 32, "parallelism": "cpu",
                   "batch_per_step": B,
                   "note": ("CPU arm: full batch-32 steps" if B == 32 else
                            f"CPU arm: each step is a batch-{B} sample of the batch-32 workload (bounded run time)")},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{args.steps} full train steps (fwd+bwd+AdamW) at batch {B}, torch CPU fp32, "
                                   f"{threads} threads of {cores} cores"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------- CUDA arm
def run_cuda(args):
    import numpy as np
    import torch
    import __graft_entry__ as ge
    rank, local_rank, world = dist_env()
    if world != args.gpus and world > 1:
        args.gpus = world
    torch.cuda.set_device(local_rank)
    use_dist = world > 1
    if use_dist:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ub = ge.load_package()
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    B = args.batch
    tr = ub.Trainer(B=B, device=local_rank, seed=1234 + rank)

    # random-init weights of the reference architecture: PyTorch default init, seed 0 (identical on every rank)
    import unet_oracle as O
    cfg = O.UNetConfig()
    flat = O.flatten_params(cfg, O.init_params(cfg, seed=0)).numpy()
    tr.set_params(flat)

    if use_dist:
        idt = torch.zeros(ub.UB_NCCL_ID_BYTES, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(ub.nccl_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        tr.attach_dp(rank, world, bytes(idt.cpu().numpy().tobytes()))

    g = torch.Generator().manual_seed(99 + rank)
    n_host = 4
    host_batches = [(torch.rand(B, 3, 64, 64, generator=g) * 2 - 1).pin_memory() for _ in range(n_host)]
    dev_batch = host_batches[0].cuda()
    stream = torch.cuda.ExternalStream(tr.stream())
    hp = dict(lr=1e-4, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0)

    def barrier():
        torch.cuda.synchronize()
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        for i in range(steps):
            fn(i)
        e1.record(stream)
        tr.sync()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if use_dist:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- device-resident throughput (`value`)
    for i in range(max(args.warmup, 3)):
        tr.train_step_device(dev_batch.data_ptr(), **hp)
    tr.sync()
    launches0 = int(ub.lib().ub_launch_count())
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ms_total = timed(lambda i: tr.train_step_device(dev_batch.data_ptr(), **hp), args.steps)
    clocks = sampler.stop() if sampler else None
    launches = int(ub.lib().ub_launch_count()) - launches0
    ms_step = ms_total / args.steps
    value = world * B / (ms_step * 1e-3)
    loss_now = tr.last_loss()
    if args.dump_outputs and rank == 0:   # before the end-to-end leg below trains further
        dump_outputs(args.dump_outputs, tr)

    # ---- end to end through the public API with HOST buffers: H2D of the batch + D2H of the loss every step
    import ctypes
    loss_c = ctypes.c_float()

    def e2e_step(i):
        # every step: announce the next pinned batch (its H2D copy then runs on the trainer's copy stream under this
        # step's kernels), H2D of this step's batch (already on its way when it was announced), 4-byte loss readback
        if not args.no_prefetch:
            tr.set_next_batch(host_batches[(i + 1) % n_host].data_ptr())
        tr.train_step_ptr(host_batches[i % n_host].data_ptr(), loss_ref=ctypes.byref(loss_c), **hp)

    for i in range(3):
        e2e_step(i)
    t_e2e = []
    barrier()
    t0 = time.perf_counter()
    for i in range(3, 3 + args.steps):
        e2e_step(i)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    e2e_ms = torch.tensor([wall * 1e3 / args.steps], device="cuda")
    if use_dist:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_value = world * B / (float(e2e_ms.item()) * 1e-3)

    # ---- live per-kernel-class timing (CUDA events around every launch, same process, same stream)
    prof = tr.profile(reps=3) if rank == 0 else None

    if rank == 0:
        pk = peaks()
        conv = prof["conv_igemm"]
        conv_tf = conv["flops"] / (conv["ms"] * 1e-3) / 1e12 if conv["ms"] > 0 else 0.0
        traffic, traffic_note = conv_traffic()
        roofline = {
            "bound": "tensor", "kernel": "igemm_conv[_ms]_kernel + igemm_conv2[_ms]_kernel + igemm_rows_kernel (3x3/1x1 conv fprop+dgrad, qkv/proj GEMMs; tcgen05)",
            "achieved": conv_tf, "peak": pk["tf_sustained"], "unit": "TFLOP/s",
            "frac": conv_tf / pk["tf_sustained"], "traffic": traffic, "traffic_note": traffic_note,
            "bytes_per_launch": conv["bytes"] / max(conv["launches"], 1),
            "peak_source": pk["source"] + ", sustained bf16",
            "flops_per_launch": conv["flops"] / max(conv["launches"], 1),
            "avg_launch_ms": conv["ms"] / max(conv["launches"], 1), "launches_per_step": conv["launches"],
            "share_of_step": conv["ms"] / prof["total_ms"],
        }
        # the other two kernel classes that carry most of the step: weight gradients (tensor) and GroupNorm (HBM)
        wg, gn = prof["wgrad_igemm"], prof["groupnorm"]
        wg_tf = wg["flops"] / (wg["ms"] * 1e-3) / 1e12 if wg["ms"] > 0 else 0.0
        gn_gbs = gn["bytes"] / (gn["ms"] * 1e-3) / 1e9 if gn["ms"] > 0 else 0.0
        roofline_more = {
            "wgrad": {"bound": "tensor", "kernel": "igemm_wgrad_kernel (tcgen05, split-K, TMA reduce-add accumulation)",
                      "achieved": wg_tf, "peak": pk["tf_sustained"], "unit": "TFLOP/s", "frac": wg_tf / pk["tf_sustained"],
                      "launches_per_step": wg["launches"], "avg_launch_ms": wg["ms"] / max(wg["launches"], 1)},
            "groupnorm": {"bound": "hbm", "kernel": "gn_apply / gn_bwd_apply_dz / gn_stats (+ gn_slab_*)",
                          "achieved": gn_gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gn_gbs / pk["hbm_gbs"],
                          "launches_per_step": gn["launches"], "avg_launch_ms": gn["ms"] / max(gn["launches"], 1),
                          "note": "algorithmic bytes / event time; most launches are latency-bound tensors of <= 4 MB "
                                  "(ncu per-kernel DRAM throughput: profiles/r02_final_hbm_kernels.txt)"},
        }
        classes = {}
        for k in ub.UB_KINDS:
            c = prof[k]
            ent = {"ms": round(c["ms"], 4), "launches": c["launches"]}
            if c["flops"] > 0 and c["ms"] > 0:
                ent["tflops"] = round(c["flops"] / (c["ms"] * 1e-3) / 1e12, 1)
            if c["bytes"] > 0 and c["ms"] > 0:
                ent["alg_gbs"] = round(c["bytes"] / (c["ms"] * 1e-3) / 1e9, 1)
            classes[k] = ent
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "train_unet default 64x64 unconditional U-Net (20494211 params, channel_mult 1-2-3-4, "
                                   "attention at 16x16 and 8x8), full train step (q-sample, fwd, MSE, bwd, AdamW)",
                       "batch_per_gpu": B, "global_batch": B * world, "parallelism": f"dp{world}",
                       "weights": "random init (PyTorch default, seed 0)", "cuda_graph": True,
                       "l2": "per-step working set (~2 GB of bf16 activations + 330 MB optimizer state) exceeds the "
                             "126 MB L2; no extra flush"},
            "clocks": clocks, "gpu_launches": launches,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": B * 3 * 64 * 64 * 4,
                    "d2h_bytes_per_step": 4, "ms_per_step": float(e2e_ms.item())},
            "roofline": roofline, "roofline_more": roofline_more, "kernel_classes": classes,
            "profile_total_ms": prof["total_ms"],
            "model_tflops": value * FLOP_PER_IMG_FWD_BWD / 1e12 / world,
            "loss_after": loss_now,
        }
        if world == 1 and not args.no_cpu_baseline:
            Bc = cpu_sample_batch(25.0, 4)
            sec, cores, threads = cpu_step_timer(Bc, 3, 1)
            line["cpu_baseline"] = {"value": Bc / sec, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": f"3 full train steps at batch {Bc}"
                                              + ("" if Bc == 32 else f" (a batch-{Bc} sample of the batch-32 workload)")
                                              + f", torch CPU fp32 oracle, {threads} threads of {cores} cores"}
            ref = reference_cuda_baseline(args)
            if ref:
                line["reference_cuda"] = ref
        if world == 1:
            line["conv_microbench"] = conv_microbench(ub, pk)
        print(json.dumps(line), flush=True)
    tr.close()
    if use_dist:
        dist.barrier()
        dist.destroy_process_group()


DUMP_SAMPLE = 1 << 22   # parameters kept in the dump: 16 MB in float32 of the 82 MB vector


def dump_outputs(out_dir, tr):
    """What the last timed step handed its caller, as float32 .npy files: the loss, the model output (B, C, H, W) and the
    updated parameters at DUMP_SAMPLE positions drawn with a fixed seed.  (The fused AdamW clears the gradients, so a
    training step returns none.)  The bench's inputs are seeded, so two builds run with the same arguments can be
    compared file by file."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    idx = np.sort(np.random.default_rng(0).choice(tr.nparams, size=min(DUMP_SAMPLE, tr.nparams), replace=False))
    arrays = {"loss": np.array([tr.last_loss()], dtype=np.float32), "output": tr.get_output(),
              "params_sample": tr.get_params()[idx]}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def conv_microbench(ub, pk):
    """The second half of BASELINE.json's metric ("conv3x3 fwd/bwd TFLOP/s vs peak", configs[1]) on a few shapes, live:
    tcgen05 conv forward / input-gradient / weight-gradient on NHWC bf16 operands resident in HBM, batch 32, CUDA
    events, L2 flushed (256 MB memset) between repetitions.  The full sweep is tools/conv_bench.py."""
    import ctypes as C
    import math
    import torch
    L = ub.lib()
    p = lambda t: C.c_void_p(t.data_ptr())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    out = []
    for (ci, co, h) in ((64, 64, 64), (128, 128, 32), (256, 256, 32), (512, 512, 64)):
        B = 32
        x = torch.randn(B, ci, h, h, device="cuda")
        w = torch.randn(co, ci, 3, 3, device="cuda") / math.sqrt(9 * ci)
        b = torch.randn(co, device="cuda")
        dout = torch.randn(B, co, h, h, device="cuda")
        dw, db = torch.empty_like(w), torch.empty_like(b)
        xb = torch.empty(B * h * h * ci, dtype=torch.bfloat16, device="cuda")
        dyb = torch.empty(B * h * h * co, dtype=torch.bfloat16, device="cuda")
        ob, dxb = torch.empty_like(dyb), torch.empty_like(xb)
        wf = torch.empty(9 * co * ci, dtype=torch.bfloat16, device="cuda")
        wd = torch.empty_like(wf)
        L.ub_nchw_to_nhwc_bf16(p(x), p(xb), B, ci, h, h)
        L.ub_nchw_to_nhwc_bf16(p(dout), p(dyb), B, co, h, h)
        L.ub_pack_conv_weight(p(w), p(wf), p(wd), ci, co, 3)
        runs = {"fwd": lambda: L.ub_conv2d_nhwc_forward(p(xb), p(wf), p(b), p(ob), B, h, h, ci, co, 3),
                "dgrad": lambda: L.ub_conv2d_nhwc_dgrad(p(dyb), p(wd), p(dxb), B, h, h, ci, co, 3),
                "wgrad": lambda: L.ub_conv2d_nhwc_wgrad(p(dyb), p(xb), p(dw), p(db), B, h, h, ci, co, 3)}
        flops = 2.0 * 9 * B * h * h * ci * co
        ent = {"shape": f"B32 {ci}->{co} @{h}x{h}", "gflop": flops / 1e9}
        for name, fn in runs.items():
            for _ in range(5):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            tot = 0.0
            for _ in range(10):
                flush.zero_()
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                tot += e0.elapsed_time(e1)
            tf = flops / (tot / 10) / 1e9
            ent[name] = {"tflops": round(tf, 1), "frac_of_burst_peak": round(tf / pk["tf_burst"], 3)}
        out.append(ent)
    return out


def kernel_source_hash():
    """sha1 over the tcgen05 conv kernel sources: profiles/*_tc_traffic.json is only valid for the kernels it was
    captured from."""
    import hashlib
    h = hashlib.sha1()
    for f in ("igemm.cu", "igemm_rows.cu", "epilogue.cuh", "ptx.cuh", "igemm.cuh"):
        with open(os.path.join(ROOT, "unet.cu_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:12]


def conv_traffic():
    """DRAM bytes per launch of the conv kernels (read + write) from the committed ncu capture of one training step
    (profiles/r02_tc_traffic.json, produced by tools/measure_all.sh + tools/traffic_summary.py, stamped with the hash of
    the kernel sources it was taken from).  (None, why) when absent or stale."""
    p = os.path.join(ROOT, "profiles", "r02_tc_traffic.json")
    try:
        with open(p) as f:
            d = json.load(f)
        stamp = d.get("_kernel_source_hash")
        if stamp != kernel_source_hash():
            return None, f"profiles/r02_tc_traffic.json was captured from kernel sources {stamp}, current {kernel_source_hash()}: stale"
        ks = [v for k, v in d.items() if k in ("igemm_conv_kernel", "igemm_conv2_kernel", "igemm_rows_kernel",
                                               "igemm_conv_ms_kernel", "igemm_conv2_ms_kernel")]
        n = sum(v["launches"] for v in ks)
        byts = sum(v["launches"] * (v["dram_read_bytes_per_launch"] + v["dram_write_bytes_per_launch"]) for v in ks)
        return (byts / n if n else None), ("DRAM bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum of one "
                                           "training step, profiles/r02_tc_traffic.json, kernel sources " + stamp +
                                           "; writes are absorbed by the L2 within the kernel); algorithmic bytes per "
                                           "launch = bytes_per_launch")
    except Exception as e:
        return None, f"no ncu traffic capture ({type(e).__name__})"


def reference_cuda_baseline(args):
    """The reference's own CUDA trainer (train_unet.cu built unmodified for sm_100 into oracle/_ref/train_unet by
    oracle/Makefile) timed for a bounded ~20 s on the same GPU: parsed from its own log lines
    (train_unet.cu:5045-5051: 'step N/... | cur time X s')."""
    exe = os.path.join(ROOT, "oracle", "_ref", "train_unet")
    # (train_unet_log10 = the same source with the log cadence literal 100 -> 10, oracle/Makefile: two log lines after
    #  30 iterations instead of 200)
    every = 100
    if os.path.exists(exe + "_log10"):
        exe, every = exe + "_log10", 10
    if not os.path.exists(exe) or args.no_reference_cuda:
        return None
    try:
        import numpy as np
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import unet_oracle as O
        with tempfile.TemporaryDirectory() as d:
            cfg = O.UNetConfig()
            flat = O.flatten_params(cfg, O.init_params(cfg, seed=0)).numpy()
            O.write_model_bin(os.path.join(d, "unet_init.bin"), cfg, flat, B=32)
            rng = np.random.default_rng(0)
            O.write_data_bin(os.path.join(d, "data.bin"), rng.uniform(-1, 1, (256, 3, 64, 64)).astype(np.float32))
            log = os.path.join(d, "log.txt")
            p = subprocess.Popen([exe, "--model_weights", "unet_init.bin", "--data_file", "data.bin", "--log_file",
                                  "log.txt"], cwd=d, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            t0 = time.time()
            pts = []
            while time.time() - t0 < (75 if every == 10 else 170):   # a log line every `every` iterations: wait for three
                time.sleep(0.5)
                if os.path.exists(log):
                    pts = []
                    for ln in open(log).read().splitlines():
                        if ln.startswith("step") and "cur time" in ln:
                            it = int(ln.split("/")[0].split()[1])
                            sec = float(ln.split("cur time")[1].split()[0])
                            pts.append((it, sec))
                    if len(pts) >= (6 if every == 10 else 2) or p.poll() is not None:
                        break
            p.kill()
            p.wait()
            what = ("reference train_unet.cu (fp32 SIMT + cuBLAS), unmodified, nvcc -O3 --use_fast_math -arch=sm_100, same "
                    "GPU, from its own 'cur time' log (CUDA-event time since its loop started, train_unet.cu:5014-5043)")
            if len(pts) >= 2:   # steady state: deltas between consecutive log lines (no cold start, no lazy mallocs)
                iv = [(b[1] - a[1]) / (b[0] - a[0]) * 1e3 for a, b in zip(pts[:-1], pts[1:])]
                sv = sorted(iv)
                ms = sv[len(sv) // 2] if len(sv) % 2 else 0.5 * (sv[len(sv) // 2 - 1] + sv[len(sv) // 2])
                cold = pts[0][1] / pts[0][0] * 1e3
                # (the reference's step time wanders from one interval to the next on a B200 box -- 220 .. 850 ms within
                #  one run, profiles/r02_reference_cuda.txt: per-call cudaMalloc / cudaFree, 46 device synchronisations
                #  per backward and a 1 GiB memset per step are host-side costs; every interval is reported)
                return {"ms_per_step": ms, "value": 32 / (ms * 1e-3), "unit": UNIT, "batch": 32,
                        "what": what + "; median of the intervals between its log lines", "iters_measured":
                        [pts[0][0], pts[-1][0]], "intervals_ms_per_step": [round(v, 1) for v in iv],
                        "ms_per_step_best_interval": round(min(iv), 1),
                        "ms_per_step_first_interval_incl_cold_start": cold}
            if pts:
                it, sec = pts[-1]
                ms = sec / it * 1e3
                return {"ms_per_step": ms, "value": 32 / (ms * 1e-3), "unit": UNIT, "batch": 32,
                        "what": what + "; cumulative over the first interval (includes cold start)", "iters_measured": it}
            return {"error": "no log line within 170 s"}
    except Exception as e:  # the comparison line is best effort
        return {"error": str(e)[:200]}
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--batch", type=int, default=32, help="per-GPU batch")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-reference-cuda", action="store_true")
    ap.add_argument("--no-prefetch", action="store_true",
                    help="end-to-end leg without ub_trainer_set_next_batch (synchronous H2D before every step)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss, model output and sampled updated parameters of the last timed step to DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        # the CPU arm sizes its batch from a timing probe, so its inputs are not the same from run to run
        ap.error("--dump-outputs applies to --impl cuda only")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
