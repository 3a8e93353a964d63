"""Generate the golden fixtures in tests/golden/ from the UNMODIFIED reference.  TEST INFRASTRUCTURE.

Needs the reference tree (``MCVD_REFERENCE_ROOT``):   python -m oracle.gen_golden [name ...]

For each small workload it instantiates the reference ``UNetMore_DDPM`` on CPU, re-randomises the
weights with the deterministic hash fill (``mcvd_b200.detfill``; seed 1234), and records
  * the forward output eps for t in {0, 37, 990} on the synthetic (x_T, cond),
  * the output of the reference ``ddpm_sampler`` / ``ddim_sampler`` / ``FPNDM_sampler`` (L = the
    workload's subsample) with per-step noise injected by patching ``torch.randn_like`` around the
    unmodified reference call,
  * the autoregressive video_gen block loop (restated; the reference's loop is entangled with
    dataset / metric code) driven by the reference sampler.
Inputs and weights are NOT stored (they regenerate bit-identically from the hash); only outputs are.
"""
from __future__ import annotations

import hashlib
import os
import sys
from unittest import mock

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from mcvd_b200 import configs, detfill          # noqa: E402
from oracle import ref_import, mcvd_oracle as O  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
T_VALUES = (0, 37, 990)


def step_noise(shape, L, tag="z"):
    return [detfill.normal(f"{tag}{i}", shape) for i in range(L - 1)]


def gen(name):
    cfg = configs.workload(name)
    net = ref_import.build_reference_net(cfg)
    _, ddpm, ddim, fpndm = ref_import.ref_models()
    B = cfg.bench_batch
    x, cond = detfill.synthetic_inputs(cfg, B)
    L = cfg.sampling.subsample
    out = {}
    with torch.no_grad():
        for t in T_VALUES:
            out[f"eps_t{t}"] = net(x, torch.full((B,), t, dtype=torch.long), cond=cond).numpy()
        zs = step_noise(x.shape, L)
        it = iter(zs)
        with mock.patch("torch.randn_like", lambda _x: next(it)):
            out["ddpm"] = ddpm(x.clone(), net, cond=cond, final_only=True, denoise=True, subsample_steps=L,
                               clip_before=True, log=False, verbose=False)[0].numpy()
        # init_prev_t warm start (t_min > 0): first randn_like call is the re-noising, then the per-step noise
        it2 = iter([detfill.normal("warm", x.shape)] + zs)
        with mock.patch("torch.randn_like", lambda _x: next(it2)):
            out["ddpm_tmin"] = ddpm(x.clone(), net, cond=cond, final_only=True, denoise=True, subsample_steps=L,
                                    clip_before=True, log=False, verbose=False, t_min=0.35)[0].numpy()
        out["ddim"] = ddim(x.clone(), net, cond=cond, final_only=True, denoise=True, subsample_steps=L,
                           clip_before=True, log=False, verbose=False)[0].numpy()
        out["fpndm"] = fpndm(x.clone(), net, cond=cond, final_only=True, subsample_steps=L,
                             clip_before=True, log=False, verbose=False)[0].numpy()
        # AR loop (runner:1501-1570 restated in the oracle) around the reference sampler
        nfp = cfg.sampling.num_frames_pred
        n_iter = -(-nfp // cfg.data.num_frames)
        inits = [detfill.normal(f"ar_init{i}", x.shape) for i in range(n_iter)]

        def sampler(x_T, c, i):
            zi = iter(step_noise(x.shape, L, tag=f"ar{i}_z"))
            with mock.patch("torch.randn_like", lambda _x: next(zi)):
                return ddpm(x_T.clone(), net, cond=c, final_only=True, denoise=True, subsample_steps=L,
                            clip_before=True, log=False, verbose=False)
        out["video"] = O.video_gen_loop(cfg, sampler, cond, inits, nfp).numpy()
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, f"{name}.npz")
    np.savez_compressed(path, **out)
    print(name, {k: v.shape for k, v in out.items()}, os.path.getsize(path) // 1024, "KiB")


def tensor_digest(t) -> np.uint64:
    """First 8 bytes of the SHA-256 of a tensor's values: pins exact equality without storing the tensor."""
    return np.frombuffer(hashlib.sha256(t.detach().cpu().contiguous().numpy().tobytes()).digest()[:8], np.uint64)[0]


def frame_table(out, X):
    """[B, K] index of the frame of ``X [B, T, C, S, S]`` that each C-channel block of ``out [B, K*C, S, S]`` is,
    -1 for an all-zero block.  ``conditioning_fn`` only slices, masks and concatenates frames, so this records its
    output exactly and independently of the values in X."""
    B, T, C = X.shape[:3]
    table = np.full((B, out.shape[1] // C), -2, np.int64)
    for b in range(B):
        for k in range(table.shape[1]):
            blk = out[b, k * C:(k + 1) * C]
            if not blk.any():
                table[b, k] = -1
            else:
                table[b, k] = next(t for t in range(T) if torch.equal(blk, X[b, t]))
    return table


def gen_reference_host():
    """``reference_host.npz``: what the CPU tests of the module layout and of ``conditioning_fn`` compare with.
    Per workload: the reference's state_dict keys and shapes, the names of its parameters (what its ``EMAHelper``
    copies by name), a digest of every re-randomised tensor and the forward output at mixed timesteps.  For the
    conditioning cases of tests/test_host_cpu.py: frame tables of the reference's outputs and its masks."""
    out = {}
    for name in ("tiny", "tiny_spade", "cfg1"):
        cfg = configs.workload(name)
        net = ref_import.build_reference_net(cfg)
        sd = net.state_dict()
        out[f"{name}_keys"] = np.array(list(sd))
        out[f"{name}_shapes"] = np.array([list(v.shape) + [-1] * (4 - v.dim()) for v in sd.values()], np.int64)
        out[f"{name}_params"] = np.array([n for n, p in net.named_parameters() if p.requires_grad])
        out[f"{name}_digest"] = np.array([tensor_digest(v) for v in sd.values()], np.uint64)
        B = cfg.bench_batch
        x, cond = detfill.synthetic_inputs(cfg, B)
        t = torch.tensor([3, 640][:B] + [77] * max(0, B - 2))
        with torch.no_grad():
            out[f"{name}_eps"] = net(x, t, cond=cond).numpy()
    R = ref_import.ref_runner()
    cfg = configs.workload("tiny")
    X = torch.arange(2 * 8 * 1 * 32 * 32, dtype=torch.float32).reshape(2, 8, 1, 32, 32)
    p, c, m = R.conditioning_fn(cfg, X, num_frames_pred=5)
    assert m is None
    out["cond_arange_pred"], out["cond_arange_cond"] = frame_table(p, X), frame_table(c, X)
    cfg.data.num_frames_future = 2
    n = cfg.data.num_frames_cond + cfg.data.num_frames + cfg.data.num_frames_future
    X = detfill.normal("clips", (6, n, cfg.data.channels, 32, 32))
    for p_cond, p_fut, sync in [(0.0, 0.0, False), (0.5, 0.0, False), (0.5, 0.5, False), (0.5, 0.5, True),
                                (0.0, 1.0, False), (0.3, 1.0, False)]:
        cfg.data.prob_mask_sync = sync
        torch.manual_seed(7)
        p, c, m = R.conditioning_fn(cfg, X, num_frames_pred=cfg.data.num_frames, prob_mask_cond=p_cond,
                                    prob_mask_future=p_fut)
        key = f"mask_{p_cond}_{p_fut}_{int(sync)}"
        out[f"{key}_pred"], out[f"{key}_cond"] = frame_table(p, X), frame_table(c, X)
        out[f"{key}_mask"] = np.zeros(0, np.int32) if m is None else m.numpy()
    u, uc, um = R.conditioning_fn(cfg, X, conditional=False)
    assert uc is None and um is None
    out["uncond_pred"] = frame_table(u, X)
    path = os.path.join(OUT, "reference_host.npz")
    np.savez_compressed(path, **out)
    print("reference_host", os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    assert ref_import.available(), "reference tree not found"
    for n in (sys.argv[1:] or ["tiny", "tiny_spade", "tiny_rgb", "cfg1", "reference_host"]):
        gen_reference_host() if n == "reference_host" else gen(n)
