#!/usr/bin/env python
"""Benchmark of the MCVD DDPM-sampling hot path on B200.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torch.distributed.run)
    python bench.py --impl reference ...                      (CPU arm: the reference algorithm on host cores)

One "step" = one full reverse-diffusion pass over one batch of clips: L network evaluations + the
final denoise evaluation + L fused updates (models/__init__.py:207-340 in the reference), i.e. one
``ddpm_sampler`` call; it produces B * num_frames frames.  With ``--ar`` a step is the whole autoregressive
``video_gen`` loop of the reference (runners/ncsn_runner.py:1501-1570): ceil(num_frames_pred / num_frames) sampler
calls with the sliding conditioning window, num_frames_pred kept frames per clip.
Default workload = BASELINE.json configs[1] ("cfg2": smmnist_DDPM_big5 + ngf=96, batch 64, subsample 100,
64x64x1, concat conditioning).
Multi-GPU: every rank owns its OWN clips (global clip ids, distinct synthetic data, noise keyed by the global
clip id), no data-path collective, and ONE NCCL all-gather of the finished frames, which is inside the e2e timed
region together with the host<->device copies.  ``--scaling weak`` (default): ``batch`` clips per GPU;
``--scaling strong``: the workload's batch split over the GPUs (BASELINE: cfg4 on 4, cfg5 on 8).

Prints ONE JSON line on rank 0 (see the keys at the bottom).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # stdout carries exactly one JSON line

import numpy as np  # noqa: E402
import torch  # noqa: E402

from mcvd_b200 import configs, detfill  # noqa: E402

METRIC = "frames/sec @100 DDPM steps, SMMNIST 64x64"
DUMP_BYTES = 64 << 20                                   # --dump-outputs size limit


def log(msg):
    if int(os.environ.get("RANK", "0")) == 0:
        print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def cpu_threads():
    """Threads for the CPU arm: every host core up to 16 (oneDNN convolutions at batch 1-8 stop scaling
    and then slow down beyond that on the 128-core GPU hosts; measured with tools/cpu_scaling.py)."""
    return int(os.environ.get("MCVD_CPU_THREADS", min(os.cpu_count() or 1, 16)))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2")
    ap.add_argument("--batch", type=int, default=0, help="clips per GPU (default: the workload's)")
    ap.add_argument("--subsample", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-psnr", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--conv", default=None, choices=[None, "umma", "umma2", "simt"])
    ap.add_argument("--ar", action="store_true", help="time the full autoregressive video_gen loop (num_frames_pred frames)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--cpu-batch", type=int, default=0, help="clips per CPU-arm step (0 = 2, or 1 when --steps > 5)")
    ap.add_argument("--psnr-steps", type=int, default=0, help="DDPM steps of the PSNR check (default: the workload's)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frames of the last timed step to DIR/frames.npy (float32) for output comparisons")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the CUDA path (--impl ours)")
    return args


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons, power = [], [], set(), []
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                              ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_min_mhz": min(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ flops
def algorithmic_gflop_per_forward(cfg) -> float:
    """conv + matmul FLOPs (2 per MAC) of ONE sample-forward on the reference graph (BASELINE.md table)."""
    from mcvd_b200 import arch
    ns = arch.build_spec(cfg)
    S = ns.image_size
    fl = 0.0

    def conv(cin, cout, r, k):
        return 2.0 * cin * cout * k * k * r * r

    fl += 2.0 * (ns.nf * ns.temb_dim + ns.temb_dim * ns.temb_dim)
    n_norms = 0
    for ms in ns.mods:
        if ms.kind == "conv3x3":
            fl += conv(ms.in_ch, ms.out_ch, ms.res, 3)
        elif ms.kind == "res":
            r_out = ms.res * 2 if ms.up else (ms.res // 2 if ms.down else ms.res)
            fl += conv(ms.in_ch, ms.out_ch, r_out, 3) + conv(ms.out_ch, ms.out_ch, r_out, 3)
            if ms.has_shortcut:
                fl += conv(ms.in_ch, ms.out_ch, r_out, 1)
            fl += 2.0 * ns.temb_dim * (2 * ms.in_ch + 2 * ms.out_ch)
            if ns.spade:
                for ch, r in ((ms.in_ch, ms.res), (ms.out_ch, r_out)):
                    fl += conv(ns.cond_ch, ns.spade_dim, r, 3) + 2 * conv(ns.spade_dim, ch, r, 3)
        elif ms.kind == "attn":
            T, C = ms.res * ms.res, ms.in_ch
            fl += 4 * 2.0 * C * C * T + 2 * 2.0 * T * T * C
        elif ms.kind == "norm" and ns.spade:
            fl += conv(ns.cond_ch, ns.spade_dim, S, 3) + 2 * conv(ns.spade_dim, ms.in_ch, S, 3)
    return fl / 1e9


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


# ------------------------------------------------------------------------------------------------ CPU arm
def _reference_root():
    """The unmodified reference tree named by MCVD_REFERENCE_ROOT or installed under baseline/_ref, if there is one."""
    for c in (os.environ.get("MCVD_REFERENCE_ROOT"), os.path.join(ROOT, "baseline", "_ref")):
        if c and os.path.exists(os.path.join(c, "models", "better", "ncsnpp_more.py")):
            return c
    return None


class CpuArm:
    """The reference's CPU implementation of the path: the UNMODIFIED reference (``UNetMore_DDPM`` +
    ``ddpm_sampler``, models/better/ncsnpp_more.py:721-770, models/__init__.py:207-340) imported in place when its
    tree is reachable, else the oracle port of the same algorithm (oracle/mcvd_oracle.py, pinned to the reference).
    One timed step = ONE FULL L-step sampler call (+ denoise) on ``batch`` clips -- no extrapolation."""

    def __init__(self, cfg, workload, batch):
        from mcvd_b200.synthetic import make_module
        self.cfg, self.B = cfg, batch
        _, _, self.sd = make_module(workload, "cpu")
        self.x, self.cond = detfill.synthetic_inputs(cfg, batch)
        self.L = cfg.sampling.subsample
        root = _reference_root()
        self.kind = "port"
        self.ref_net = None
        if root is not None:
            try:
                os.environ["MCVD_REFERENCE_ROOT"] = root
                from oracle import ref_import
                if ref_import.available():
                    net = ref_import.build_reference_net(cfg)
                    net.load_state_dict(self.sd, strict=False)
                    self.ref_net, self.ref_sampler, self.kind = net.eval(), ref_import.ref_models()[1], "reference"
            except Exception as e:                               # any import problem: the port is always there
                log(f"reference tree at {root} not usable ({type(e).__name__}: {e}); timing the oracle port")
        self.threads, self.thread_scan = self._pick_threads()

    def forward(self):
        t = torch.full((self.B,), 500, dtype=torch.long)
        with torch.no_grad():
            if self.ref_net is not None:
                return self.ref_net(self.x, t, cond=self.cond)
            from oracle import mcvd_oracle as O
            return O.unet_forward(self.cfg, self.sd, self.x, t, self.cond)

    def _pick_threads(self):
        """oneDNN convolutions at batch 1-2 stop scaling well before 128 threads on the GPU hosts (and get slower):
        time one forward at a few thread counts and keep the fastest."""
        if os.environ.get("MCVD_CPU_THREADS"):
            n = int(os.environ["MCVD_CPU_THREADS"])
            torch.set_num_threads(n)
            return n, {}
        ncpu = os.cpu_count() or 1
        scan = {}
        self_threads = sorted({min(ncpu, 8), min(ncpu, 16), min(ncpu, 32), min(ncpu, 64), ncpu})
        for n in self_threads:
            torch.set_num_threads(n)
            self.forward()
            t0 = time.perf_counter()
            self.forward()
            scan[n] = time.perf_counter() - t0
            # ascending scan, stop at the first clear regression: on the 128-core GPU hosts one forward takes 0.08 s
            # at 16 threads and 48 s at 128 -- trying every count would cost minutes of the arm's budget
            if len(scan) >= 2 and scan[n] > 1.3 * min(scan.values()):
                break
        best = min(scan, key=scan.get)
        torch.set_num_threads(best)
        return best, {str(k): round(v, 3) for k, v in scan.items()}

    def sample(self):
        """one full sampler call; returns seconds"""
        torch.manual_seed(1234)
        t0 = time.perf_counter()
        with torch.no_grad():
            if self.ref_net is not None:
                self.ref_sampler(self.x.clone(), self.ref_net, cond=self.cond, final_only=True, denoise=True,
                                 subsample_steps=self.L, clip_before=True, verbose=False, log=False)
            else:
                from oracle import mcvd_oracle as O
                fn = lambda xx, tt, cc: O.unet_forward(self.cfg, self.sd, xx, tt, cc)
                O.ddpm_sample(fn, O.make_schedule(self.cfg), self.x.clone(), self.cond, self.L, True, True)
        return time.perf_counter() - t0

    def describe(self, dt):
        import platform
        cpu = platform.processor() or "unknown CPU"
        try:
            for line in open("/proc/cpuinfo"):
                if line.startswith("model name"):
                    cpu = line.split(":", 1)[1].strip()
                    break
        except OSError:
            pass
        impl = ("unmodified reference UNetMore_DDPM + ddpm_sampler" if self.kind == "reference"
                else "oracle port of the reference (oracle/mcvd_oracle.py)")
        return (f"each step = one full {self.L}-step DDPM sampler call (+ denoise) of the {impl} on {self.B} clip(s) "
                f"({dt:.1f} s), {self.threads} threads of {os.cpu_count()} on {cpu}; threads picked from one forward at "
                f"each of {self.thread_scan}")


def run_reference_arm(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # clips per step: 2 for short runs, 1 when the driver asks for many steps (a step is a FULL sampler call, ~8 s per
    # clip on the GPU hosts: K = 20 then stays within a few minutes); frames/s is per-clip work either way
    if not args.cpu_batch:
        args.cpu_batch = 2 if args.steps <= 5 else 1
    arm = CpuArm(cfg, args.workload, args.cpu_batch)
    log(f"CPU arm: {arm.kind}, {arm.threads} threads, scan {arm.thread_scan}, {args.cpu_batch} clip(s) per step")
    for i in range(args.warmup):
        arm.forward()                                            # warm-up steps are single forwards (allocator, oneDNN)
    dts = [arm.sample() for _ in range(args.steps)]
    dt = statistics.mean(dts)
    frames = args.cpu_batch * cfg.data.num_frames
    v = frames / dt
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {describe(cfg)}", "clips_per_step": args.cpu_batch,
                       "note": "same network, sampler, steps and frame counts as the GPU arm; the CPU arm runs "
                               f"{args.cpu_batch} clip(s) per step instead of {cfg.bench_batch} (a 64-clip CPU step takes "
                               "tens of minutes); frames/s is per-clip work either way"},
            "cpu_baseline": {"value": v, "unit": "frames/s", "cores": arm.threads, "kind": arm.kind,
                             "sample": arm.describe(dt)},
            "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def describe(cfg):
    d, m = cfg.data, cfg.model
    return (f"{d.image_size}x{d.image_size}x{d.channels}, frames {d.num_frames}+{d.num_frames_cond} cond, ngf {m.ngf}, "
            f"ch_mult {list(m.ch_mult)}, {'SPADE' if getattr(m, 'spade', False) else 'concat'} conditioning, "
            f"DDPM subsample {cfg.sampling.subsample}")


# ------------------------------------------------------------------------------------------------ main
def main():
    args = parse()
    cfg = configs.workload(args.workload)
    if args.subsample:
        cfg.sampling.subsample = args.subsample
    if args.impl == "reference":
        return run_reference_arm(args, cfg)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py (impl=ours) needs a CUDA device; there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.conv:
        os.environ["MCVD_CONV"] = args.conv

    from mcvd_b200.synthetic import make_module
    from mcvd_b200 import samplers, runner, lib
    cfg, net, sd = make_module(args.workload, dev)
    if args.subsample:
        cfg.sampling.subsample = args.subsample
    L = cfg.sampling.subsample
    C, F, S = cfg.data.channels, cfg.data.num_frames, cfg.data.image_size
    nfp = cfg.sampling.num_frames_pred if args.ar else F           # kept frames per clip and step
    n_iter = -(-nfp // F) if args.ar else 1                         # sampler calls per step
    # clips: weak scaling = `batch` clips on every GPU; strong scaling = the workload's batch split over the GPUs
    if args.scaling == "strong":
        n_clips = args.batch or cfg.bench_batch
        lo, hi = runner.shard_range(n_clips, rank, world)
    else:
        B_rank = args.batch or cfg.bench_batch
        n_clips = B_rank * world
        lo, hi = rank * B_rank, (rank + 1) * B_rank
    B = hi - lo
    assert B > 0, f"rank {rank} has no clips ({n_clips} clips over {world} GPUs)"
    # every clip has its own synthetic data, generated for the GLOBAL clip index (same clip on any GPU count)
    x_all, cond_all = detfill.synthetic_inputs(cfg, n_clips)
    x_host, cond_host = x_all[lo:hi].contiguous().pin_memory(), cond_all[lo:hi].contiguous().pin_memory()
    x_dev, cond_dev = x_host.to(dev), cond_host.to(dev)
    out_host = torch.empty((n_clips, C * nfp, S, S), dtype=torch.float32).pin_memory() if rank == 0 else None
    kw = dict(final_only=True, denoise=True, subsample_steps=L, clip_before=True, verbose=False, log=False)

    def generate(i, xd, cd):
        """this rank's clips: one sampler call, or the whole AR loop; frames in [0, 1]"""
        if args.ar:
            return runner.video_gen_clips(cfg, net, cd, nfp, clip_offset=lo, philox_seed=1234 + i,
                                          init_fn=lambda k, shape: xd if k == 0 else torch.randn(shape, device=dev),
                                          sampler=samplers.ddpm_sampler, sampler_kwargs=dict(subsample_steps=L))
        gen = samplers.ddpm_sampler(xd, net, cond=cd, philox_seed=1234 + i, clip_offset=lo, **kw)[-1]
        return runner.inverse_data_transform(cfg, gen)

    def step_resident(i):
        return generate(i, x_dev, cond_dev)

    def step_e2e(i):
        xd = x_host.to(dev, non_blocking=True)
        cd = cond_host.to(dev, non_blocking=True)
        frames = generate(i, xd, cd)
        allf = runner.gather_clips(frames, n_clips, rank, world)      # the one collective of the path (NCCL all-gather)
        if rank == 0:
            out_host.copy_(allf.reshape(out_host.shape), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return out_host

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, K):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms

    log(f"module built; clips {lo}..{hi} of {n_clips} (B={B}), L={L}, {n_iter} sampler call(s) per step; warm-up x{args.warmup}")
    for i in range(args.warmup):
        step_resident(i)
        torch.cuda.synchronize()
        log(f"warm-up step {i} done")
    launches_per_step = samplers.ddpm_sampler.last_launches * n_iter
    clocks = ClockSampler(local)
    clocks.start()
    ms = timed(step_resident, args.steps)
    clk = clocks.stop()
    frames_per_step = n_clips * nfp
    value = frames_per_step * args.steps / (ms / 1e3)
    log(f"resident: {ms / args.steps:.1f} ms/step -> {value:.1f} frames/s")
    for i in range(min(args.warmup, 1)):
        step_e2e(i)
    clocks2 = ClockSampler(local)                                    # the e2e region is clock-sampled too
    clocks2.start()
    ms_e2e = timed(step_e2e, args.steps)
    clk_e2e = clocks2.stop()
    e2e_val = frames_per_step * args.steps / (ms_e2e / 1e3)
    log(f"e2e: {ms_e2e / args.steps:.1f} ms/step -> {e2e_val:.1f} frames/s")
    if rank == 0 and args.dump_outputs:
        # what the last timed e2e step returned: every clip's frames on the host, [clips, C * frames, S, S] in [0, 1];
        # above DUMP_BYTES only every k-th clip is written, the same clips on every run with the same arguments
        frames = out_host.numpy()
        stride = -(-len(frames) // (DUMP_BYTES // frames[0].nbytes))
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "frames.npy"), frames[::stride])
        log(f"wrote {args.dump_outputs}/frames.npy: every {stride} clip(s) of {tuple(frames.shape)}")

    gf = algorithmic_gflop_per_forward(cfg)
    pk, pk_src = peaks()
    P = net.engine().program(B)
    calls = (L + 1) * n_iter                                        # network evaluations per clip and step
    gen_frames = n_clips * F * n_iter                               # frames generated (the AR loop keeps nfp of them)
    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f32 (fp16 hi/lo split on tcgen05, fp32 accumulate)", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {describe(cfg)}", "clips_per_gpu": B, "global_clips": n_clips,
                   "mode": (f"autoregressive video_gen: {n_iter} sampler calls per step, {nfp} frames kept of "
                            f"{F * n_iter} generated per clip" if args.ar else "one ddpm_sampler call per step"),
                   "parallelism": f"clip-sharded x{world} (distinct clips per rank, global clip ids), no data-path "
                                  f"collective; one NCCL all-gather of the finished frames inside the e2e region",
                   "l2": "working set (weights 4x%.0f MB + GBs of activations per forward) exceeds the 126 MB L2; no flush needed"
                         % (sum(p.numel() for p in net.parameters()) / 1e6),
                   "conv_backend": net.engine().conv_mode, "noise": "in-kernel Philox4x32-10 keyed by global clip id"},
        "e2e": {"value": e2e_val, "unit": "frames/s", "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": (x_host.numel() + cond_host.numel()) * 4 * world,
                "d2h_bytes_per_step": n_clips * C * nfp * S * S * 4,
                "allgather_bytes_per_rank_per_step": (B * C * nfp * S * S * 4) if world > 1 else 0,
                "clocks": clk_e2e},
        "gpu_launches": int(launches_per_step * args.steps),
        "clocks": clk,
        "frames_generated_per_s": gen_frames * args.steps / (ms / 1e3),
        "flops": {"algorithmic_gflop_per_sample_forward": gf,
                  "algorithmic_tflop_per_kept_frame": gf * calls / nfp / 1e3,
                  "whole_path_achieved_tflops": value * gf * calls / nfp / 1e3 / world,
                  "whole_path_frac_of_bf16_peak": value * gf * calls / nfp / 1e3 / world / pk["bf16_tflops_sustained"],
                  "note": "tensor work executed = 3x algorithmic (fp16 hi/lo split for fp32 parity)"},
    }

    if rank == 0 and not args.no_roofline:
        line["roofline"] = roofline(net, P, B, cfg, pk, pk_src)
    if rank == 0 and world == 1 and not args.no_psnr:
        log("PSNR check (CUDA path vs oracle on CPU, 1 clip)")
        line["psnr_vs_oracle_db"] = psnr_check(cfg, net, sd, dev, steps=args.psnr_steps or min(L, 100))
        line["psnr_steps"] = args.psnr_steps or min(L, 100)
        log(f"psnr {line['psnr_vs_oracle_db']:.1f} dB")
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        log("CPU baseline: one full sampler call on the host cores")
        arm = CpuArm(cfg, args.workload, 1)
        arm.forward()
        dt = arm.sample()
        line["cpu_baseline"] = {"value": cfg.data.num_frames / dt, "unit": "frames/s", "cores": arm.threads,
                                "kind": arm.kind, "sample": arm.describe(dt)}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def roofline(net, P, B, cfg, pk, pk_src):
    """Per-op CUDA-event timing of the lowered program (2 forwards after a warm-up one), on the launch
    stream; the dominant kernel is the tcgen05 implicit-GEMM conv (k_conv_umma)."""
    from mcvd_b200 import lib
    eng = net.engine()
    n = len(P.step_ops)
    stream = torch.cuda.current_stream().cuda_stream
    step_ptr = ctypes.cast(P.step_arr, ctypes.POINTER(lib.McvdOp))
    sz = ctypes.sizeof(lib.McvdOp)

    def op_ptr(i):
        return ctypes.cast(ctypes.addressof(P.step_arr) + i * sz, ctypes.POINTER(lib.McvdOp))

    eng.run_step(P)
    torch.cuda.synchronize()
    reps = 2
    tot = {}
    flops_umma = 0.0
    for rep in range(reps):
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
        evs[0].record()
        for i in range(n):
            lib.check(lib.load().mcvd_run_program(op_ptr(i), 1, ctypes.c_void_p(stream)), "run_program")
            evs[i + 1].record()
        torch.cuda.synchronize()
        for i in range(n):
            op = P.step_ops[i]
            ms = evs[i].elapsed_time(evs[i + 1])
            k = tot.setdefault(op.kind, [0.0, 0])
            k[0] += ms
            k[1] += 2 if op.kind == lib.OP_ATTENTION_UMMA else 1   # pre-split + attention kernels
            if op.kind in (lib.OP_CONV_UMMA, lib.OP_CONV_UMMA2) and rep == 0:
                flops_umma += 2.0 * op.B * op.H * op.W * (op.C0 + op.C1) * op.Cout * op.i0 * op.i0
    names = {v: k for k, v in vars(lib).items() if k.startswith("OP_")}
    per_kind = {names[k][3:].lower(): {"ms_per_forward": v[0] / reps, "launches_per_forward": v[1] // reps}
                for k, v in sorted(tot.items(), key=lambda kv: -kv[1][0])}
    total_ms = sum(v[0] for v in tot.values()) / reps
    out = {"bound": "tensor", "unit": "TFLOP/s", "peak": pk["bf16_tflops_sustained"],
           "peak_source": f"{pk_src} cuBLAS bf16 sustained (MEASURED_PEAKS.json)", "traffic": None,
           "per_kind": per_kind, "forward_ms_sum_of_kernels": total_ms}
    conv_kind = lib.OP_CONV_UMMA if lib.OP_CONV_UMMA in tot else lib.OP_CONV_UMMA2
    if conv_kind in tot:
        n_umma = tot[conv_kind][1] // reps
        # algorithmic HBM bytes of the kernel: every conv reads its input(s) and writes its output once (fp32),
        # plus residual and the packed weights
        alg_bytes = 0.0
        for op in P.step_ops:
            if op.kind == conv_kind:
                px = op.B * op.H * op.W
                alg_bytes += 4.0 * px * (op.C0 + op.C1 + op.C2 + op.C3 + op.Cout * (2 if op.aux0 else 1))
                alg_bytes += 4.0 * op.Cout * ((op.C0 + op.C1) * op.i0 * op.i0 + op.C2 + op.C3)
        tpath = os.path.join(ROOT, "profiles", "ncu_conv_umma_traffic.json")
        if os.path.exists(tpath) and "cfg2" in getattr(cfg, "workload", "") and B == 64:
            tj = json.load(open(tpath))
            out["traffic"] = tj["dram_bytes_per_launch_mean"]
            out["traffic_note"] = (f"mean dram__bytes_read+write per conv launch ({tj['kernel']}) from the committed ncu pass "
                                   f"({tj['launches_per_forward']} launches, {tj['dram_bytes_per_forward'] / 1e9:.2f} GB per "
                                   f"forward); algorithmic {alg_bytes / 1e9:.2f} GB per forward")
        out["algorithmic_bytes_per_launch"] = alg_bytes / max(n_umma, 1)
        ms_umma = tot[conv_kind][0] / reps
        ach = flops_umma / (ms_umma / 1e3) / 1e12
        out.update(kernel=("k_conv_umma (3x3) + k_conv1x1_umma (1x1)" if conv_kind == lib.OP_CONV_UMMA
                           else "k_conv_umma2 (cta_group::2)") + " (tcgen05 implicit-GEMM convs, all conv launches of one forward)",
                   achieved=ach, frac=ach / pk["bf16_tflops_sustained"], executed_tflops=3 * ach,
                   executed_frac=3 * ach / pk["bf16_tflops_sustained"],
                   kernel_share_of_forward=ms_umma / total_ms,
                   algorithmic_gflop_per_forward_in_kernel=flops_umma / 1e9)
    else:
        ms_simt = tot.get(lib.OP_CONV_SIMT, [0.0, 0])[0] / reps
        out.update(kernel="k_conv_simt", achieved=None, frac=None, kernel_share_of_forward=ms_simt / max(total_ms, 1e-9))
    return out


def psnr_check(cfg, net, sd, dev, B=1, steps=None):
    """Full L-step DDPM sampling of one clip with injected noise: CUDA path vs the oracle (CPU)."""
    from mcvd_b200 import samplers
    from oracle import mcvd_oracle as O
    L = steps or cfg.sampling.subsample
    x, cond = detfill.synthetic_inputs(cfg, B, seed=77)
    zs = [detfill.normal(f"pz{i}", x.shape, seed=77) for i in range(L - 1)]
    out = samplers.ddpm_sampler(x.to(dev), net, cond=cond.to(dev), final_only=True, denoise=True, subsample_steps=L,
                                noise_list=[z.to(dev) for z in zs])[0].cpu()
    torch.set_num_threads(cpu_threads())
    fn = lambda xx, tt, cc: O.unet_forward(cfg, sd, xx, tt, cc)
    ref = O.ddpm_sample(fn, O.make_schedule(cfg), x.clone(), cond, L, True, True, noise=zs)[0]
    to01 = lambda a: ((a + 1) / 2).clamp(0, 1)
    return O.psnr01(to01(out), to01(ref))


if __name__ == "__main__":
    # stdout must carry exactly ONE JSON line: libraries (NCCL's version banner, torch warnings) write to fd 1
    # behind Python's back, so fd 1 is pointed at stderr for the whole run and restored only for the result.
    sys.stdout.flush()
    _real_stdout = os.dup(1)
    os.dup2(2, 1)
    _buf = []
    _print = print

    def print(*a, **k):  # noqa: A001  (module-level print used by main() for the JSON line)
        if k.get("file") in (None, sys.stdout):
            _buf.append(" ".join(str(x) for x in a))
        else:
            _print(*a, **k)

    try:
        main()
    finally:
        sys.stdout.flush()
        os.dup2(_real_stdout, 1)
        os.close(_real_stdout)
        for line in _buf:
            _print(line, flush=True)
