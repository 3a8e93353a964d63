#!/usr/bin/env python
"""Cost of the noise options on the B200: frames/s of one AR iteration of ``runner.video_gen_clips`` (one 100-step
DDPM sampler call, B clips x num_frames frames) with each option off and on.

    python tools/bench_noise_options.py [--rounds R] [--warmup W]

  * cfg2 (concat conditioning, B = 64): model.gamma off / on (Gamma per-step noise and Gamma x_T; video_gen_clips
    passes gamma from the config, as the reference's runner does);
  * cfg2 and cfg3 (SPADE, B = 32): model.noise_in_cond off / on.  On SPADE nets noise_in_cond moves the gamma/beta
    convolutions from once per sampler call into every network evaluation, so cfg3 pays them 101 times.

All variants share their network weights, live in one process and are timed in alternation (round-robin, CUDA
events around each call, ``--warmup`` untimed calls per variant first, as bench.py does).  Noise is drawn in-kernel
(Philox), so the timed region holds no host-side random numbers.  Prints one JSON line with the median frames/s of
every variant, the spread, and the card name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from mcvd_b200 import configs, detfill, runner  # noqa: E402
from mcvd_b200.synthetic import make_module  # noqa: E402


def card():
    """(name, power limit in W) of cuda:0, read now"""
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(q.splitlines()[0])
    except Exception:
        power = None
    return name, power


def variant(workload, **model):
    cfg = configs.workload(workload)
    for k, v in model.items():
        setattr(cfg.model, k, v)
    cfg, net, _ = make_module(cfg, "cuda:0")
    _, cond = detfill.synthetic_inputs(cfg, cfg.bench_batch)
    return cfg, net, cond.cuda()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_noise_options: needs a CUDA device")
    name, power = card()
    variants = {
        "cfg2": variant("cfg2"),
        "cfg2_gamma": variant("cfg2", gamma=True),
        "cfg2_noise_in_cond": variant("cfg2", noise_in_cond=True),
        "cfg3": variant("cfg3"),
        "cfg3_noise_in_cond": variant("cfg3", noise_in_cond=True),
    }

    def call(cfg, net, cond, i):
        return runner.video_gen_clips(cfg, net, cond, cfg.data.num_frames, philox_seed=1000 + i, init_seed=2000 + i)

    times = {k: [] for k in variants}
    for k, (cfg, net, cond) in variants.items():
        for w in range(args.warmup):
            call(cfg, net, cond, w)
    torch.cuda.synchronize()
    for r in range(args.rounds):
        for k, (cfg, net, cond) in variants.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = call(cfg, net, cond, r)
            e1.record()
            torch.cuda.synchronize()
            assert torch.isfinite(out).all(), k
            times[k].append(e0.elapsed_time(e1) / 1e3)
    res = {}
    for k, (cfg, net, cond) in variants.items():
        frames = cfg.bench_batch * cfg.data.num_frames
        fps = [frames / t for t in times[k]]
        res[k] = {"frames_per_s": statistics.median(fps), "min": min(fps), "max": max(fps), "batch": cfg.bench_batch,
                  "steps": cfg.sampling.subsample}
    rel = {"cfg2_gamma_vs_off": res["cfg2_gamma"]["frames_per_s"] / res["cfg2"]["frames_per_s"],
           "cfg2_noise_in_cond_vs_off": res["cfg2_noise_in_cond"]["frames_per_s"] / res["cfg2"]["frames_per_s"],
           "cfg3_noise_in_cond_vs_off": res["cfg3_noise_in_cond"]["frames_per_s"] / res["cfg3"]["frames_per_s"]}
    print(json.dumps({"metric": "frames/s, one 100-step DDPM AR iteration of video_gen_clips", "gpu": name,
                      "power_limit_w": power, "rounds": args.rounds, "warmup": args.warmup, "variants": res,
                      "ratio": rel}))


if __name__ == "__main__":
    main()
