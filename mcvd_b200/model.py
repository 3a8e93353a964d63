"""Drop-in replacement for the reference ``UNetMore_DDPM`` (``models/better/ncsnpp_more.py:721-770``).

Same constructor argument (the config Namespace), same ``forward(x, y, cond=None, cond_mask=None)``,
same ``state_dict`` keys and shapes (``unet.all_modules.{i}...``, buffers ``betas / alphas /
alphas_prev / unet.sigmas``, plus ``k / k_cum / theta_t`` with ``gamma``) so reference checkpoints load with
``load_state_dict`` and
``EMAHelper.ema`` can copy weights in by name (``models/ema.py:23-28``).  The modules below hold
parameters only; all arithmetic runs in the CUDA library through a lowered op program
(``mcvd_b200/program.py``).  There is no PyTorch or CPU fallback: calling ``forward`` without the
library or off-GPU raises.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import numpy as np
import torch
import torch.nn as nn

from . import arch


def _variance_scaling_uniform(shape, scale=1.0, in_axis=1, out_axis=0):
    """DDPM 'fan_avg uniform' initialiser (same rule as reference layers.py:43-79)."""
    scale = 1e-10 if scale == 0 else scale
    receptive = int(np.prod(shape)) / shape[in_axis] / shape[out_axis]
    fan_in, fan_out = shape[in_axis] * receptive, shape[out_axis] * receptive
    limit = math.sqrt(3.0 * scale / ((fan_in + fan_out) / 2.0))
    return (torch.rand(*shape) * 2.0 - 1.0) * limit


class _Affine(nn.Module):
    """weight/bias holder (nn.Linear, nn.Conv2d or affine nn.GroupNorm in the reference)."""

    def __init__(self, wshape, init_scale=1.0, norm=False):
        super().__init__()
        if norm:
            self.weight = nn.Parameter(torch.ones(wshape))
            self.bias = nn.Parameter(torch.zeros(wshape))
        else:
            self.weight = nn.Parameter(_variance_scaling_uniform(wshape, init_scale))
            self.bias = nn.Parameter(torch.zeros(wshape[0]))


class _NIN(nn.Module):
    def __init__(self, cin, cout, init_scale=0.1):
        super().__init__()
        self.W = nn.Parameter(_variance_scaling_uniform((cin, cout), init_scale))
        self.b = nn.Parameter(torch.zeros(cout))


class _Spade(nn.Module):
    """MySPADE parameters (layerspp.py:148-150): mlp_shared.0, mlp_gamma, mlp_beta (3x3 convs)."""

    def __init__(self, ch, cond_ch, spade_dim):
        super().__init__()
        self.mlp_shared = nn.Sequential(_Affine((spade_dim, cond_ch, 3, 3)))
        self.mlp_gamma = _Affine((ch, spade_dim, 3, 3))
        self.mlp_beta = _Affine((ch, spade_dim, 3, 3))


class _ActNorm(nn.Module):
    """get_act_norm parameters (layerspp.py:486-516)."""

    def __init__(self, ch, temb_dim, spade, cond_ch, spade_dim):
        super().__init__()
        if temb_dim is not None:
            self.Dense_0 = _Affine((2 * ch, temb_dim))
        if spade:
            self.Norm_0 = _Spade(ch, cond_ch, spade_dim)
        elif temb_dim is None:
            self.Norm_0 = _Affine(ch, norm=True)   # affine GroupNorm of the final norm
        else:
            self.Norm_0 = nn.Module()              # param-free GroupNorm


class _ResBlock(nn.Module):
    def __init__(self, ms: arch.ModSpec, ns: arch.NetSpec):
        super().__init__()
        self.actnorm0 = _ActNorm(ms.in_ch, ns.temb_dim, ns.spade, ns.cond_ch, ns.spade_dim)
        self.Conv_0 = _Affine((ms.out_ch, ms.in_ch, 3, 3))
        self.actnorm1 = _ActNorm(ms.out_ch, ns.temb_dim, ns.spade, ns.cond_ch, ns.spade_dim)
        self.Conv_1 = _Affine((ms.out_ch, ms.out_ch, 3, 3), init_scale=0.0)
        if ms.has_shortcut:
            self.Conv_2 = _Affine((ms.out_ch, ms.in_ch, 1, 1))


class _AttnBlock(nn.Module):
    def __init__(self, ch):
        super().__init__()
        self.GroupNorm_0 = _Affine(ch, norm=True)
        self.NIN_0 = _NIN(ch, ch)
        self.NIN_1 = _NIN(ch, ch)
        self.NIN_2 = _NIN(ch, ch)
        self.NIN_3 = _NIN(ch, ch, init_scale=0.0)


class _UNet(nn.Module):
    def __init__(self, config, ns: arch.NetSpec):
        super().__init__()
        mods = []
        for ms in ns.mods:
            if ms.kind == "linear":
                mods.append(_Affine((ms.out_ch, ms.in_ch)))
            elif ms.kind == "conv3x3":
                last = ms.idx == len(ns.mods) - 1
                mods.append(_Affine((ms.out_ch, ms.in_ch, 3, 3), init_scale=0.0 if last else 1.0))
            elif ms.kind == "res":
                mods.append(_ResBlock(ms, ns))
            elif ms.kind == "attn":
                mods.append(_AttnBlock(ms.in_ch))
            elif ms.kind == "norm":
                mods.append(_ActNorm(ms.in_ch, None, ns.spade, ns.cond_ch, ns.spade_dim))
        self.all_modules = nn.ModuleList(mods)
        m = config.model
        self.register_buffer("sigmas", torch.linspace(m.sigma_begin, m.sigma_end, m.num_classes))


class UNetMore_DDPM(nn.Module):
    """B200-native score network with the reference's module interface."""

    def __init__(self, config):
        super().__init__()
        why = arch.check_supported(config)
        if why is not None:
            raise NotImplementedError(f"mcvd_b200 does not accelerate this configuration: {why}")
        self.config = config
        self.version = getattr(config.model, "version", "DDPM").upper()
        self.spec = arch.build_spec(config)
        self.unet = _UNet(config, self.spec)
        m = config.model
        betas = torch.linspace(m.sigma_begin, m.sigma_end, m.num_classes)       # models/__init__.py:24-26
        alphas = torch.cumprod(1 - betas.flip(0), 0).flip(0)                    # ncsnpp_more.py:737-739
        self.register_buffer("betas", betas)
        self.register_buffer("alphas", alphas)
        self.register_buffer("alphas_prev", torch.cat([alphas[1:], torch.tensor([1.0])]))
        self.schedule = "linear"
        self.gamma = bool(getattr(m, "gamma", False))
        if self.gamma:                       # Gamma diffusion noise, ncsnpp_more.py:744-749 (same names and order)
            self.theta_0 = 0.001
            self.register_buffer("k", betas / (alphas * (self.theta_0 ** 2)))
            self.register_buffer("k_cum", torch.cumsum(self.k.flip(0), 0).flip(0))
            self.register_buffer("theta_t", torch.sqrt(alphas) * self.theta_0)
        self.noise_in_cond = bool(getattr(m, "noise_in_cond", False))
        self.type = getattr(config.model, "type", "v1")
        self._engine = None

    # -- engine management -----------------------------------------------------------------------
    def engine(self):
        """The lowered CUDA program cache for this module (created on first use)."""
        if self._engine is None:
            from .program import Engine
            self._engine = Engine(self)
        return self._engine

    def _apply(self, fn, *a, **k):
        r = super()._apply(fn, *a, **k)
        self._engine = None          # device / dtype change invalidates packed weights and buffers
        return r

    def _replicate_for_data_parallel(self):
        """``torch.nn.DataParallel`` shallow-copies the module per GPU (reference runners/ncsn_runner.py:1377);
        every replica must lower and pack for ITS device, not share device 0's engine."""
        r = super()._replicate_for_data_parallel()
        r._engine = None
        return r

    def forward(self, x, y, cond=None, cond_mask=None, cond_noise=None):
        """eps = net(x_t, t, cond).  x [B, C*F, S, S] fp32 NCHW, y [B] (int64 or float), cond
        [B, C*Fc, S, S] or None.  ``cond_mask`` only matters for ``cond_emb=True`` nets, which are not
        built by this class (reference ncsnpp_more.py:283-287).

        ``noise_in_cond`` nets first diffuse cond to each clip's timestep y (ncsnpp_more.py:753-766), so y must hold
        integer labels, as the reference's ``alphas[labels]`` requires.  The noise is ``cond_noise`` when given (the
        normalised noise, shaped like cond), else fresh from torch's RNG: ``torch.randn_like(cond)``, or on a
        ``gamma`` net a Gamma draw made in-kernel under a seed taken from torch's generator."""
        if not x.is_cuda and not (self._engine is not None and self._engine.backend is not None):
            raise RuntimeError("mcvd_b200.UNetMore_DDPM runs on CUDA (sm_100a) only; no CPU fallback exists")
        philox = None
        if self.noise_in_cond and cond is not None:
            check_labels(self, y)
            if cond_noise is None:
                if self.gamma:
                    philox = (int(torch.randint(0, 2 ** 62, (1,)).item()), 0)
                else:
                    cond_noise = torch.randn_like(cond)
        return self.engine().forward(x, y, cond, cond_noise=cond_noise, cond_philox=philox)


def check_labels(net, y):
    """``alphas[labels]`` of the reference's noise_in_cond forward (ncsnpp_more.py:757-759): floating-point labels
    raise (only integer tensors index), and so do labels outside the schedule."""
    if not torch.is_tensor(y) or torch.is_floating_point(y):
        raise IndexError("noise_in_cond: the labels index alphas[labels], so they must be an integer tensor "
                         f"(got {y.dtype if torch.is_tensor(y) else type(y).__name__})")
    n = net.alphas.numel()
    if y.numel() and (int(y.min()) < 0 or int(y.max()) >= n):
        raise IndexError(f"noise_in_cond: labels must lie in [0, {n})")


def get_model(config):
    """Same contract as reference ``runners/ncsn_runner.py:180-195``: module on ``config.device``."""
    return UNetMore_DDPM(config).to(config.device)
