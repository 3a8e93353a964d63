"""CPU oracle for the MCVD DDPM-sampling hot path.  TEST INFRASTRUCTURE ONLY.

This file is a plain PyTorch fp32 *restatement* of the reference algorithm (voletiv/mcvd-pytorch
@ 451da2e) for the path BASELINE.json names: the conditional NCSN++ ("UNetMore") score network,
the DDPM / DDIM / F-PNDM reverse-diffusion loops and the autoregressive ``video_gen`` outer loop.
It is functional (driven by a reference-format ``state_dict``), runs on the CPU, and exists so the
CUDA path can be checked on the GPU box where ``/root/reference`` does not exist.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference``
legs may import this module.  The product package ``mcvd_b200`` never does.

Pinning: the reference has NO tests or golden vectors for this path (SURVEY.md section 4/8c), so the
oracle is pinned against the reference *itself*: the committed fixtures in ``tests/golden/`` are produced by
``oracle/gen_golden.py`` from the unmodified reference, imported in place, and the tests compare with them.

Every function cites the reference file:line it restates (paths relative to the reference root).
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional

import numpy as np
import torch
import torch.nn.functional as F

Tensor = torch.Tensor


# ----------------------------------------------------------------------------- schedule
def make_schedule(config) -> Dict[str, Tensor]:
    """betas / alphas / alphas_prev buffers.

    ``models/__init__.py:16-35`` (get_sigmas, 'linear': linspace(sigma_begin, sigma_end, T)) and
    ``models/better/ncsnpp_more.py:735-739``: alphas = flip(cumprod(1 - flip(betas))); index 0 is the
    noisiest level; alphas_prev = [alphas[1:], 1].
    """
    m = config.model
    assert getattr(m, "sigma_dist", "linear") == "linear"
    betas = torch.linspace(m.sigma_begin, m.sigma_end, m.num_classes)
    alphas = torch.cumprod(1 - betas.flip(0), 0).flip(0)
    alphas_prev = torch.cat([alphas[1:], torch.tensor([1.0])])
    return dict(betas=betas, alphas=alphas, alphas_prev=alphas_prev)


# ----------------------------------------------------------------------------- small pieces
def num_groups(ch: int) -> int:
    """GroupNorm group rule, ``models/better/layerspp.py:474-477`` (also :212-214, :127-130)."""
    g = min(ch // 4, 32)
    while ch % g != 0:
        g -= 1
    return g


def timestep_embedding(t: Tensor, dim: int) -> Tensor:
    """``models/better/layers.py:504-518`` get_timestep_embedding (max_positions = 10000)."""
    half = dim // 2
    freq = torch.exp(torch.arange(half, dtype=torch.float32) * -(math.log(10000) / (half - 1)))
    e = t.float()[:, None] * freq[None, :]
    e = torch.cat([torch.sin(e), torch.cos(e)], dim=1)
    if dim % 2 == 1:
        e = F.pad(e, (0, 1))
    return e


def fir_taps(up: bool) -> Tensor:
    """4x4 FIR taps: outer([1,3,3,1]) / 64, times 4 when upsampling.

    ``models/better/up_or_down_sampling.py:182-189`` (_setup_kernel) and :220-222 / :252-254.
    """
    k = np.outer(np.asarray([1, 3, 3, 1], np.float32), np.asarray([1, 3, 3, 1], np.float32))
    k /= k.sum()
    if up:
        k = k * 4.0
    return torch.from_numpy(k.astype(np.float32))


def fir_upsample(x: Tensor) -> Tensor:
    """upsample_2d(factor 2): zero-insert, pad (2,1), 4x4 FIR.

    ``up_or_down_sampling.py:196-225`` -> ``op/upfirdn2d.py:163-204`` (upfirdn2d_native).  Restated
    as a transposed-convolution-free gather: insert zeros, pad, correlate with the flipped taps.
    """
    B, C, H, W = x.shape
    z = x.new_zeros(B, C, 2 * H, 2 * W)
    z[:, :, ::2, ::2] = x
    z = F.pad(z, (2, 1, 2, 1))
    k = torch.flip(fir_taps(True), [0, 1]).view(1, 1, 4, 4)
    out = F.conv2d(z.reshape(B * C, 1, 2 * H + 3, 2 * W + 3), k)
    return out.reshape(B, C, 2 * H, 2 * W)


def fir_downsample(x: Tensor) -> Tensor:
    """downsample_2d(factor 2): pad (1,1), 4x4 FIR, keep every 2nd sample.

    ``up_or_down_sampling.py:228-258`` -> ``op/upfirdn2d.py:163-204``.
    """
    B, C, H, W = x.shape
    z = F.pad(x, (1, 1, 1, 1))
    k = torch.flip(fir_taps(False), [0, 1]).view(1, 1, 4, 4)
    out = F.conv2d(z.reshape(B * C, 1, H + 2, W + 2), k)[:, :, ::2, ::2]
    return out.reshape(B, C, H // 2, W // 2)


def silu(x: Tensor) -> Tensor:
    """``models/better/layers.py:29-31``: get_act always returns nn.SiLU()."""
    return x * torch.sigmoid(x)


class _P:
    """state_dict view with a key prefix."""

    def __init__(self, sd, prefix):
        self.sd, self.prefix = sd, prefix

    def __getitem__(self, k):
        return self.sd[self.prefix + k]

    def has(self, k):
        return (self.prefix + k) in self.sd

    def sub(self, k):
        return _P(self.sd, self.prefix + k)


def spade_norm(p: _P, x: Tensor, cond: Tensor) -> Tensor:
    """MySPADE.forward, ``models/better/layerspp.py:152-173`` (2-D path).

    param-free GroupNorm(eps 1e-6) ; nearest-resize cond ; a = SiLU(conv3x3(cond)) ;
    out = normalized * (1 + conv3x3_gamma(a)) + conv3x3_beta(a).
    """
    C = x.shape[1]
    normalized = F.group_norm(x, num_groups(C), None, None, 1e-6)
    seg = F.interpolate(cond, size=x.shape[-2:], mode="nearest")
    a = silu(F.conv2d(seg, p["mlp_shared.0.weight"], p["mlp_shared.0.bias"], padding=1))
    gamma = F.conv2d(a, p["mlp_gamma.weight"], p["mlp_gamma.bias"], padding=1)
    beta = F.conv2d(a, p["mlp_beta.weight"], p["mlp_beta.bias"], padding=1)
    return normalized * (1 + gamma) + beta


def act_norm(p: _P, x: Tensor, temb: Optional[Tensor], cond: Optional[Tensor], spade: bool) -> Tensor:
    """get_act_norm.forward, ``models/better/layerspp.py:518-549`` (2-D path).

    with emb: [scale, shift] = chunk(Dense_0(SiLU(temb)), 2); y = Norm(x) * (1 + scale) + shift;
    Norm = GroupNorm(affine=False, eps=1e-5) or MySPADE.  Without emb (final norm): affine GroupNorm
    (or MySPADE).  Then SiLU.
    """
    C = x.shape[1]
    if spade:
        n = spade_norm(p.sub("Norm_0."), x, cond)
    elif p.has("Norm_0.weight"):
        n = F.group_norm(x, num_groups(C), p["Norm_0.weight"], p["Norm_0.bias"], 1e-5)
    else:
        n = F.group_norm(x, num_groups(C), None, None, 1e-5)
    if temb is not None and p.has("Dense_0.weight"):
        e = F.linear(silu(temb), p["Dense_0.weight"], p["Dense_0.bias"])[:, :, None, None]
        scale, shift = torch.chunk(e, 2, dim=1)
        n = n * (1 + scale) + shift
    return silu(n)


def resblock(p: _P, x: Tensor, temb: Tensor, cond: Optional[Tensor], spade: bool,
             up: bool, down: bool) -> Tensor:
    """ResnetBlockBigGANppGN / ...SPADE forward, ``models/better/layerspp.py:595-624, 675-705``.

    h = actnorm0(x); FIR-resample BOTH h and x when up/down; h = Conv_0(h); h = actnorm1(h);
    dropout is identity in eval; h = Conv_1(h); x = Conv_2(x) (1x1) iff it exists; (x + h) / sqrt(2).
    """
    h = act_norm(p.sub("actnorm0."), x, temb, cond, spade)
    if up:
        h, x = fir_upsample(h), fir_upsample(x)
    elif down:
        h, x = fir_downsample(h), fir_downsample(x)
    h = F.conv2d(h, p["Conv_0.weight"], p["Conv_0.bias"], padding=1)
    h = act_norm(p.sub("actnorm1."), h, temb, cond, spade)
    h = F.conv2d(h, p["Conv_1.weight"], p["Conv_1.bias"], padding=1)
    if p.has("Conv_2.weight"):
        x = F.conv2d(x, p["Conv_2.weight"], p["Conv_2.bias"])
    return (x + h) / np.sqrt(2.0)


def nin(p: _P, x: Tensor) -> Tensor:
    """NIN.forward, ``models/better/layers.py:541-544``: per-pixel x @ W[in,out] + b."""
    y = torch.einsum("bchw,cd->bdhw", x, p["W"]) + p["b"][None, :, None, None]
    return y


def attnblock(p: _P, x: Tensor, n_head_channels: int) -> Tensor:
    """AttnBlockpp.forward, ``models/better/layerspp.py:230-249``.

    GroupNorm(affine, eps 1e-6); q,k,v = NIN_{0,1,2}; heads are contiguous channel blocks;
    softmax over all H*W keys of (q.k) * Ch^-0.5; NIN_3; (x + h) / sqrt(2).
    """
    B, C, H, W = x.shape
    heads = 1 if C < n_head_channels else C // n_head_channels
    if n_head_channels == -1:
        heads = 1
    h = F.group_norm(x, num_groups(C), p["GroupNorm_0.weight"], p["GroupNorm_0.bias"], 1e-6)
    q, k, v = nin(p.sub("NIN_0."), h), nin(p.sub("NIN_1."), h), nin(p.sub("NIN_2."), h)
    Ch = C // heads
    q = q.reshape(B * heads, Ch, H * W)
    k = k.reshape(B * heads, Ch, H * W)
    v = v.reshape(B * heads, Ch, H * W)
    w = torch.einsum("bct,bcs->bts", q, k) * (int(Ch) ** (-0.5))
    w = F.softmax(w, dim=-1)
    o = torch.einsum("bts,bcs->bct", w, v).reshape(B, C, H, W)
    o = nin(p.sub("NIN_3."), o)
    return (x + o) / np.sqrt(2.0)


# ----------------------------------------------------------------------------- the network
@torch.no_grad()
def unet_forward(config, sd: Dict[str, Tensor], x: Tensor, t: Tensor, cond: Optional[Tensor] = None,
                 taps: Optional[Dict[int, Tensor]] = None) -> Tensor:
    """UNetMore_DDPM.forward -> NCSNpp.forward / SPADE_NCSNpp.forward (2-D, positional embedding).

    ``models/better/ncsnpp_more.py:753-770, 251-392, 590-718``.  ``sd`` uses the reference key names
    (``unet.all_modules.{i}...``).  ``taps`` (optional) receives the output of every module index.
    """
    m = config.model
    spade = bool(getattr(m, "spade", False))
    nf, ch_mult, nrb = m.ngf, m.ch_mult, m.num_res_blocks
    attn_res = list(m.attn_resolutions)
    nhc = m.n_head_channels
    R = len(ch_mult)
    idx = [0]

    def mod():
        p = _P(sd, f"unet.all_modules.{idx[0]}.")
        idx[0] += 1
        return p

    def rec(h):
        if taps is not None:
            taps[idx[0] - 1] = h
        return h

    if cond is not None and not spade:
        x = torch.cat([x, cond], dim=1)                      # ncsnpp_more.py:256-257
    temb = timestep_embedding(t, nf)                         # :273
    p = mod(); temb = F.linear(temb, p["weight"], p["bias"])           # :278
    p = mod(); temb = F.linear(silu(temb), p["weight"], p["bias"])     # :280
    p = mod(); h = rec(F.conv2d(x, p["weight"], p["bias"], padding=1))  # :294
    hs = [h]
    for lvl in range(R):                                     # :296-315
        for _ in range(nrb):
            h = rec(resblock(mod(), hs[-1], temb, cond, spade, False, False))
            if h.shape[-1] in attn_res:
                h = rec(attnblock(mod(), h, nhc))
            hs.append(h)
        if lvl != R - 1:
            h = rec(resblock(mod(), hs[-1], temb, cond, spade, False, True))
            hs.append(h)
    h = hs[-1]                                               # :320-338
    h = rec(resblock(mod(), h, temb, cond, spade, False, False))
    h = rec(attnblock(mod(), h, nhc))
    h = rec(resblock(mod(), h, temb, cond, spade, False, False))
    for lvl in reversed(range(R)):                           # :342-371
        for _ in range(nrb + 1):
            h = rec(resblock(mod(), torch.cat([h, hs.pop()], dim=1), temb, cond, spade, False, False))
        if h.shape[-1] in attn_res:
            h = rec(attnblock(mod(), h, nhc))
        if lvl != 0:
            h = rec(resblock(mod(), h, temb, cond, spade, True, False))
    assert not hs
    h = rec(act_norm(mod(), h, None, cond, spade))           # :375
    p = mod(); h = rec(F.conv2d(h, p["weight"], p["bias"], padding=1))  # :379
    assert not any(k.startswith(f"unet.all_modules.{idx[0]}.") for k in sd), "module count mismatch"
    return h


# ----------------------------------------------------------------------------- samplers
def _subsample(sched, subsample_steps):
    """``models/__init__.py:228-240``: skip = T // L; steps = range(0, T, skip); re-derive betas."""
    alphas, alphas_prev, betas = sched["alphas"], sched["alphas_prev"], sched["betas"]
    steps = np.arange(len(betas))
    if subsample_steps is not None and subsample_steps < len(alphas):
        skip = len(alphas) // subsample_steps
        steps = torch.tensor(list(range(0, len(alphas), skip)))
        alphas = alphas.index_select(0, steps)
        alphas_prev = torch.cat([alphas[1:], torch.tensor([1.0])])
        betas = 1.0 - torch.div(alphas, alphas_prev)
    return steps, alphas, alphas_prev, betas


@torch.no_grad()
def ddpm_sample(net, sched, x: Tensor, cond=None, subsample_steps=None, denoise=True, clip_before=True,
                noise: Optional[List[Tensor]] = None, just_beta=False, final_only=True, t_min=-1,
                warm_noise: Optional[Tensor] = None):
    """ddpm_sampler, ``models/__init__.py:207-340`` (t_min<=0, gamma=False path).

    ``net(x, labels, cond)`` is the score network.  ``noise`` is a list with one tensor per step that
    adds noise (L-1 entries); when None, torch.randn_like is used as in the reference (:324).
    ``t_min > 0`` is the ``init_prev_t`` warm start (:269-280): steps with ``step < t_min * len(alphas)`` are
    skipped (``alphas`` being the SUBSAMPLED schedule, as written) and x is first noised to the level of
    the first kept step with ``warm_noise``.
    """
    steps, alphas, alphas_prev, betas = _subsample(sched, subsample_steps)
    L = len(steps)
    images = []
    x_transf = False
    for i, step in enumerate(steps):
        if step < t_min * len(alphas):                                                   # :269-270
            continue
        if not x_transf and t_min > 0:                                                   # :272-279
            z0 = warm_noise if warm_noise is not None else torch.randn_like(x)
            x = alphas[i].sqrt() * x + (1 - alphas[i]).sqrt() * z0
        x_transf = True
        c_beta, c_alpha, c_alpha_prev = betas[i], alphas[i], alphas_prev[i]
        labels = (step * torch.ones(x.shape[0])).long()                                  # :283
        grad = net(x, labels, cond)                                                      # :284
        x0 = (1 / c_alpha.sqrt()) * (x - (1 - c_alpha).sqrt() * grad)                    # :287
        if clip_before:
            x0 = x0.clip_(-1, 1)                                                         # :289
        x = (c_alpha_prev.sqrt() * c_beta / (1 - c_alpha)) * x0 + \
            ((1 - c_beta).sqrt() * (1 - c_alpha_prev) / (1 - c_alpha)) * x               # :290
        if not final_only:
            images.append(x.clone())
        if i + 1 == L:                                                                   # :311-313
            continue
        z = noise[i] if noise is not None else torch.randn_like(x)
        if just_beta:
            x = x + c_beta.sqrt() * z
        else:
            x = x + ((1 - c_alpha_prev) / (1 - c_alpha) * c_beta).sqrt() * z             # :328
    if denoise:                                                                          # :331-333
        last = ((L - 1) * torch.ones(x.shape[0])).long()
        x = x - (1 - alphas[-1]).sqrt() * net(x, last, cond)
        if not final_only:
            images.append(x.clone())
    return x.unsqueeze(0) if final_only else torch.stack(images)


@torch.no_grad()
def ddim_sample(net, sched, x: Tensor, cond=None, subsample_steps=None, denoise=True, clip_before=True,
                final_only=True):
    """ddim_sampler, ``models/__init__.py:103-203``: x = sqrt(a_prev) x0 + sqrt(1-a_prev) eps."""
    steps, alphas, alphas_prev, betas = _subsample(sched, subsample_steps)
    L = len(steps)
    images = []
    for i, step in enumerate(steps):
        c_alpha, c_alpha_prev = alphas[i], alphas_prev[i]
        labels = (step * torch.ones(x.shape[0])).long()
        grad = net(x, labels, cond)
        x0 = (1 / c_alpha.sqrt()) * (x - (1 - c_alpha).sqrt() * grad)                    # :163
        if clip_before:
            x0 = x0.clip_(-1, 1)
        x = c_alpha_prev.sqrt() * x0 + (1 - c_alpha_prev).sqrt() * grad                  # :166
        if not final_only:
            images.append(x.clone())
    if denoise:                                                                          # :194-196
        last = ((L - 1) * torch.ones(x.shape[0])).long()
        x = x - (1 - alphas[-1]).sqrt() * net(x, last, cond)
        if not final_only:
            images.append(x.clone())
    return x.unsqueeze(0) if final_only else torch.stack(images)


def _pndm_transfer(x, t, t_next, et, alphas_cump, clip_before):
    """``models/pndm.py:19-34`` transfer (DDIM-form update with the +1-offset lookup)."""
    at = alphas_cump[t.long() + 1].view(-1, 1, 1, 1)
    at_next = alphas_cump[t_next.long() + 1].view(-1, 1, 1, 1)
    x_delta = (at_next - at) * ((1 / (at.sqrt() * (at.sqrt() + at_next.sqrt()))) * x -
                                1 / (at.sqrt() * (((1 - at_next) * at).sqrt() + ((1 - at) * at_next).sqrt())) * et)
    x_next = x + x_delta
    if clip_before:
        x_next = x_next.clip_(-1, 1)
    return x_next


@torch.no_grad()
def fpndm_sample(net, sched, x: Tensor, cond=None, subsample_steps=None, clip_before=True, final_only=True):
    """FPNDM_sampler + pndm.gen_order_4 / runge_kutta, ``models/__init__.py:39-99``, ``models/pndm.py:3-52``.

    Replicated as written (README flags F-PNDM as "might be broken"): alphas looked up through a
    flipped copy with a +1 offset, steps_next = [-1] + steps[:-1], fractional mid-timesteps fed to the
    network (the sinusoidal embedding sees the float, the alpha lookup truncates), no denoise call.
    """
    alphas = sched["alphas"]
    alphas_old = alphas.flip(0)                                                          # :58
    skip = len(alphas) // subsample_steps
    steps = list(range(0, len(alphas), skip))
    steps_next = [-1] + steps[:-1]                                                       # :63
    ets: List[Tensor] = []
    images = []
    B = x.shape[0]
    for i in range(len(steps)):
        t = (steps[i] * torch.ones(B)).long()
        t_next = (steps_next[i] * torch.ones(B)).long()
        t_list = [t, (t + t_next) / 2, t_next]                                           # pndm.py:42
        if len(ets) > 2:                                                                 # pndm.py:44-47
            e = net(x, t, cond)
            ets.append(e)
            noise = (1 / 24) * (55 * ets[-1] - 59 * ets[-2] + 37 * ets[-3] - 9 * ets[-4])
        else:                                                                            # runge_kutta :3-17
            e1 = net(x, t_list[0], cond)
            ets.append(e1)
            x2 = _pndm_transfer(x, t_list[0], t_list[1], e1, alphas_old, clip_before)
            e2 = net(x2, t_list[1], cond)
            x3 = _pndm_transfer(x, t_list[0], t_list[1], e2, alphas_old, clip_before)
            e3 = net(x3, t_list[1], cond)
            x4 = _pndm_transfer(x, t_list[0], t_list[2], e3, alphas_old, clip_before)
            e4 = net(x4, t_list[2], cond)
            noise = (1 / 6) * (e1 + 2 * e2 + 2 * e3 + e4)
        x = _pndm_transfer(x, t, t_next, noise, alphas_old, clip_before)
        if not final_only:
            images.append(x.clone())
    return x.unsqueeze(0) if final_only else torch.stack(images)


# ----------------------------------------------------------------------------- AR outer loop
def conditioning_split(config, X: Tensor, num_frames_pred: int):
    """conditioning_fn (prob_mask_* = 0, no future frames), ``runners/ncsn_runner.py:104-147``."""
    S = config.data.image_size
    c = config.data.num_frames_cond
    pred = X[:, c:c + num_frames_pred].reshape(len(X), -1, S, S)
    cond = X[:, :c].reshape(len(X), -1, S, S)
    return pred, cond, None


@torch.no_grad()
def video_gen_loop(config, sampler, cond: Tensor, init_noise: List[Tensor], num_frames_pred: int) -> Tensor:
    """Autoregressive block loop of NCSNRunner.video_gen, ``runners/ncsn_runner.py:1501-1570``.

    ``sampler(x_T, cond, i_iter) -> [1, B, C*F, S, S]``; ``init_noise[i]`` is the fresh z drawn for AR
    iteration i (:1476, :1551).  Returns ``clamp((pred + 1) / 2, 0, 1)`` of the first ``num_frames_pred``
    frames (inverse_data_transform, ``datasets/__init__.py:252-261``).
    """
    C, Fr, Fc = config.data.channels, config.data.num_frames, config.data.num_frames_cond
    n_iter = math.ceil(num_frames_pred / Fr)
    preds = []
    for i in range(n_iter):
        gen = sampler(init_noise[i], cond, i)[-1]
        gen = gen.reshape(gen.shape[0], C * Fr, config.data.image_size, config.data.image_size)
        preds.append(gen)
        if i == n_iter - 1:
            continue
        cond = torch.cat([cond[:, C * Fr:], gen[:, C * max(0, Fr - Fc):]], dim=1)        # :1537-1539
    pred = torch.cat(preds, dim=1)[:, :C * num_frames_pred]
    return torch.clamp((pred + 1.0) / 2.0, 0.0, 1.0)


def psnr01(a: Tensor, b: Tensor) -> float:
    """PSNR on [0,1] images as the reference computes it: 10 log10(1 / MSE) (``runner:1588, 2197``)."""
    mse = torch.mean((a.double() - b.double()) ** 2).item()
    return float("inf") if mse == 0 else 10.0 * math.log10(1.0 / mse)
