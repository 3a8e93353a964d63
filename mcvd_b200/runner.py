"""Sampling slice of the reference runner: conditioning, the autoregressive block loop, clip sharding.

Restates (does not copy) ``runners/ncsn_runner.py``: ``conditioning_fn`` (:104-147), the AR loop of
``NCSNRunner.video_gen`` (:1501-1570) and ``get_sampler`` (:2702-2714); the dataset, metric, gif and
checkpoint-sweep code around them is out of scope (SURVEY.md section 8).

Multi-GPU: the reference wraps the network in ``torch.nn.DataParallel`` (:1377) and re-broadcasts all
weights on every one of the 101 x n_iter network calls.  Here every clip (batch element) is
independent through the whole AR x diffusion loop, so rank r owns clips [r*B/G, (r+1)*B/G), runs with
its own weight copy and ZERO communication, and the ranks meet in exactly one NCCL all-gather of the
finished frames (``gather_clips``).
"""
from __future__ import annotations

import math
from typing import Callable, List, Optional, Tuple

import torch

from .samplers import get_sampler


def data_transform(config, X):
    """x -> 2x - 1 for ``rescaled`` data (reference datasets/__init__.py:235-249, sampling-relevant part)."""
    if getattr(config.data, "rescaled", True):
        return 2 * X - 1.0
    return X


def inverse_data_transform(config, X):
    """clamp((x + 1) / 2, 0, 1) (reference datasets/__init__.py:252-261)."""
    if getattr(config.data, "rescaled", True):
        X = (X + 1.0) / 2.0
    return torch.clamp(X, 0.0, 1.0)


def conditioning_fn(config, X, num_frames_pred=0, prob_mask_cond=0.0, prob_mask_future=0.0, conditional=True):
    """Split ``X [B, T, C, S, S]`` into (frames to predict, conditioning frames, cond_mask).

    Same contract as reference ``runners/ncsn_runner.py:104-147`` including the Bernoulli masking of
    past / future frames used by the paper's "general" models.
    """
    S = config.data.image_size
    if not conditional:
        return X.reshape(len(X), -1, S, S), None, None
    n_cond = config.data.num_frames_cond
    n_train = config.data.num_frames
    n_future = getattr(config.data, "num_frames_future", 0)
    pred_frames = X[:, n_cond:n_cond + num_frames_pred].reshape(len(X), -1, S, S)
    cond_frames = X[:, :n_cond].reshape(len(X), -1, S, S)
    cond_mask = None
    if prob_mask_cond > 0.0:
        keep = torch.rand(X.shape[0], device=X.device) > prob_mask_cond
        cond_frames = keep.reshape(-1, 1, 1, 1) * cond_frames
        cond_mask = keep.to(torch.int32)
    if n_future > 0:
        if prob_mask_future == 1.0:
            fut = torch.zeros(len(X), config.data.channels * n_future, S, S)
        else:
            fut = X[:, n_cond + n_train:n_cond + n_train + n_future].reshape(len(X), -1, S, S)
            if prob_mask_future > 0.0:
                if getattr(config.data, "prob_mask_sync", False):
                    fmask = cond_mask
                else:
                    fmask = torch.rand(X.shape[0], device=X.device) > prob_mask_future
                fut = fmask.reshape(-1, 1, 1, 1) * fut
        cond_frames = torch.cat([cond_frames, fut.to(cond_frames.device)], dim=1)
    return pred_frames, cond_frames, cond_mask


def shard_range(n_clips: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous clip range owned by ``rank`` (first ranks take the remainder)."""
    base, rem = divmod(n_clips, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


@torch.no_grad()
def video_gen_clips(config, scorenet, cond: torch.Tensor, num_frames_pred: Optional[int] = None,
                    init_fn: Optional[Callable[[int, Tuple[int, ...]], torch.Tensor]] = None,
                    sampler=None, sampler_kwargs=None, clip_offset: int = 0, philox_seed: Optional[int] = None,
                    noise_fn: Optional[Callable[[int], List[torch.Tensor]]] = None,
                    init_seed: Optional[int] = None) -> torch.Tensor:
    """Autoregressive block generation for the clips in ``cond`` (reference runner:1501-1570).

    Each iteration samples ``num_frames`` frames, appends them, slides the conditioning window
    ``cond <- cat(cond[:, C*F:], gen[:, C*max(0, F - Fc):])`` (:1537-1539) and draws a fresh init.
    Returns ``inverse_data_transform(pred)[:, :C*num_frames_pred]`` on the input device.
    ``init_fn(i, shape)`` supplies x_T of AR iteration i (default ``torch.randn``, :1476/:1551; for a ``gamma``
    config the centred Gamma draw of :1471-1474, made in-kernel keyed by the global clip id under ``init_seed``, or a
    seed from torch's generator); ``noise_fn(i)`` optionally supplies the per-step noise list (parity tests).
    """
    from .samplers import gamma_init
    C, F, Fc = config.data.channels, config.data.num_frames, config.data.num_frames_cond
    S = config.data.image_size
    nfp = num_frames_pred if num_frames_pred is not None else config.sampling.num_frames_pred
    one_at_a_time = getattr(config.sampling, "one_frame_at_a_time", False)
    n_iter = nfp if one_at_a_time else math.ceil(nfp / F)
    sampler = sampler or get_sampler(config)
    kw = dict(final_only=True, denoise=config.sampling.denoise,
              subsample_steps=getattr(config.sampling, "subsample", None),
              clip_before=getattr(config.sampling, "clip_before", True), verbose=False, log=False,
              t_min=getattr(config.sampling, "init_prev_t", -1), gamma=getattr(config.model, "gamma", False))
    kw.update(sampler_kwargs or {})
    B = cond.shape[0]
    shape = (B, C * F, S, S)
    preds = []
    warm = (getattr(config.sampling, "init_prev_t", -1) or -1) > 0
    gen = None
    for i in range(n_iter):
        if warm and i > 0:
            x_T = gen                                    # init_prev_t > 0: restart from the previous block (:1513)
        else:
            if init_fn is not None:
                x_T = init_fn(i, shape)
            elif getattr(config.model, "gamma", False):
                seed = init_seed if init_seed is not None else int(torch.randint(0, 2 ** 62, (1,)).item())
                x_T = gamma_init(scorenet, shape, seed + 7919 * (i + 1), clip_offset)
            else:
                x_T = torch.randn(shape, device=cond.device)
        extra = {}
        if noise_fn is not None:
            extra["noise_list"] = noise_fn(i)
        elif philox_seed is not None:
            # one Philox stream per (clip, AR iteration, step): fold the AR iteration into the seed
            extra.update(philox_seed=philox_seed + 7919 * (i + 1), clip_offset=clip_offset)
        gen = sampler(x_T.to(cond.device), scorenet, cond=cond, **kw, **extra)[-1].reshape(shape)
        preds.append(gen)
        if i == n_iter - 1:
            continue
        if one_at_a_time:
            cond = torch.cat([cond[:, C:], gen[:, :C]], dim=1)
        else:
            cond = torch.cat([cond[:, C * F:], gen[:, C * max(0, F - Fc):]], dim=1)
    pred = torch.cat(preds, dim=1)[:, :C * nfp]
    return inverse_data_transform(config, pred)


def gather_clips(local: torch.Tensor, n_clips: int, rank: int, world: int, group=None) -> torch.Tensor:
    """The one collective of the path: all-gather every rank's finished frames (NCCL over NVLink).

    Shards may differ by one clip, so each rank pads to the largest shard, all-gathers into one flat
    buffer and the padding is dropped on reassembly.
    """
    import torch.distributed as dist
    if world == 1:
        return local
    sizes = [shard_range(n_clips, r, world) for r in range(world)]
    mx = max(hi - lo for lo, hi in sizes)
    pad = torch.zeros((mx,) + tuple(local.shape[1:]), device=local.device, dtype=local.dtype)
    pad[:local.shape[0]] = local
    out = torch.empty((world * mx,) + tuple(local.shape[1:]), device=local.device, dtype=local.dtype)
    dist.all_gather_into_tensor(out, pad.contiguous(), group=group)
    parts = [out[r * mx:r * mx + (hi - lo)] for r, (lo, hi) in enumerate(sizes)]
    return torch.cat(parts, dim=0)


@torch.no_grad()
def video_gen_sharded(config, scorenet, cond_all: torch.Tensor, rank: int, world: int, philox_seed: int = 1234,
                      init_seed: int = 1234, **kw) -> torch.Tensor:
    """Clip-sharded ``video_gen``: this rank generates its clips, then one all-gather.

    Initial noise, per-step noise and conditioning noise (``noise_in_cond``) are keyed by the GLOBAL clip index so
    the result is independent of the sharding (world size 1 == world size G, bit for bit).
    """
    n = cond_all.shape[0]
    lo, hi = shard_range(n, rank, world)
    dev = cond_all.device if cond_all.is_cuda else torch.device("cuda", torch.cuda.current_device())
    cond = cond_all[lo:hi].to(dev)

    def init_fn(i, shape):
        # per-clip generators: clip g of AR iteration i always sees the same x_T
        outs = []
        for g in range(lo, hi):
            gen = torch.Generator(device="cpu")
            gen.manual_seed(init_seed * 1000003 + g * 1009 + i)
            outs.append(torch.randn(shape[1:], generator=gen))
        return torch.stack(outs).to(dev) if outs else torch.empty((0,) + tuple(shape[1:]), device=dev)

    if getattr(config.model, "gamma", False):
        init_fn = None                                   # Gamma x_T, drawn in-kernel per global clip id
    local = video_gen_clips(config, scorenet, cond, init_fn=init_fn, clip_offset=lo, philox_seed=philox_seed,
                            init_seed=init_seed, **kw)
    return gather_clips(local, n, rank, world)


# ---------------------------------------------------------------------------------------------------------------
# evaluation of generated clips on the GPU (SURVEY.md section 8f rows 2 and 3)
# ---------------------------------------------------------------------------------------------------------------
def frame_metrics(config, pred: torch.Tensor, real: torch.Tensor) -> torch.Tensor:
    """Per-frame MSE and SSIM of generated clips, on the GPU: float64 [B, frames, 2].

    Replaces the reference's per-frame CPU loop over PIL images (runners/ncsn_runner.py:1581-1600).  ``pred`` and
    ``real`` are [B, C*frames, S, S] in [0, 1] (``inverse_data_transform`` output).  MovingMNIST-style datasets get the
    reference's rounding before the grey conversion (:1596-1599)."""
    from . import lib
    C, S = config.data.channels, config.data.image_size
    B, CF = pred.shape[0], pred.shape[1]
    dev = pred.device
    if dev.type != "cuda":
        raise RuntimeError("mcvd_b200.runner.frame_metrics runs on CUDA tensors only (no CPU fallback)")
    p = pred.contiguous().float()
    r = real.to(dev).contiguous().float()
    out = torch.empty(B, CF // C, 2, dtype=torch.float64, device=dev)
    op = lib.McvdOp()
    op.kind, op.B, op.H, op.W, op.C0, op.i0 = lib.OP_FRAME_METRICS, B, S, S, C, CF // C
    name = str(getattr(config.data, "dataset", "")).upper()
    op.flags = lib.F_ROUND if name in ("STOCHASTICMOVINGMNIST", "MOVINGMNIST") else 0
    op.src0, op.src1, op.dst = p.data_ptr(), r.data_ptr(), out.data_ptr()
    with torch.cuda.device(dev):
        lib.run_program(lib.make_ops([op]), 1, torch.cuda.current_stream(dev).cuda_stream)
    return out


def best_of_repeats(per_frame: torch.Tensor, preds_per_test: int):
    """(mse, psnr, ssim) per test clip: video metric = mean over frames, then the best of the clip's
    ``preds_per_test`` samples (reference runners/ncsn_runner.py:1602-1604, 2194-2196)."""
    vid_mse = per_frame[..., 0].mean(1)
    vid_ssim = per_frame[..., 1].mean(1)
    mse = vid_mse.reshape(-1, preds_per_test).min(-1).values
    psnr = (10 * torch.log10(1 / vid_mse)).reshape(-1, preds_per_test).max(-1).values
    ssim = vid_ssim.reshape(-1, preds_per_test).max(-1).values
    return mse, psnr, ssim


@torch.no_grad()
def evaluate_clips(config, scorenet, X: torch.Tensor, preds_per_test: Optional[int] = None,
                   num_frames_pred: Optional[int] = None, **gen_kw):
    """One test batch of the reference's ``video_gen`` (runners/ncsn_runner.py:1392-1395, 1463-1470, 1501-1609): every
    test clip is repeated ``preds_per_test`` times (``repeat_interleave``, the reference's collate function), each
    repeat is sampled with its own noise, and the per-clip metrics keep the best repeat.  ``X`` is [B, T, C, S, S] in
    [0, 1].  Returns (frames [B*p, C*nfp, S, S] in [0, 1], dict of per-clip mse / psnr / ssim tensors)."""
    p = preds_per_test if preds_per_test is not None else getattr(config.sampling, "preds_per_test", 1)
    nfp = num_frames_pred if num_frames_pred is not None else config.sampling.num_frames_pred
    X = X.repeat_interleave(p, dim=0)
    real, cond, _ = conditioning_fn(config, data_transform(config, X), num_frames_pred=nfp,
                                    prob_mask_cond=getattr(config.data, "prob_mask_cond", 0.0))
    dev = next(scorenet.parameters()).device
    frames = video_gen_clips(config, scorenet, cond.to(dev), nfp, **gen_kw)
    real01 = inverse_data_transform(config, real.to(dev))
    per_frame = frame_metrics(config, frames, real01)
    mse, psnr, ssim = best_of_repeats(per_frame, p)
    return frames, {"mse": mse, "psnr": psnr, "ssim": ssim, "per_frame": per_frame}
