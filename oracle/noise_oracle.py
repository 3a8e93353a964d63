"""CPU oracle of the reference's noise options, ``model.gamma`` and ``model.noise_in_cond``.  TEST INFRASTRUCTURE ONLY.

A plain PyTorch fp32 restatement, like ``oracle/mcvd_oracle.py`` (whose network and samplers it reuses), of:
  * the Gamma schedule buffers, ``models/better/ncsnpp_more.py:744-749``;
  * the conditioning noise of ``UNetMore_DDPM.forward``, ``ncsnpp_more.py:753-766``;
  * the reference's map from a Gamma draw to the noise sigma multiplies, ``models/__init__.py:148-151, 274-277,
    319-322`` and ``ncsnpp_more.py:762-765``;
  * the DDIM sampler with the ``t_min`` warm start, ``models/__init__.py:103-203``.
With the normalised noise injected, the Gamma samplers (``gamma=True``) are the normal ones: they differ only in how
the noise is drawn.  The product package ``mcvd_b200`` never imports this module.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from oracle import mcvd_oracle as O

Tensor = torch.Tensor
THETA_0 = 0.001


def make_schedule(config) -> Dict[str, Tensor]:
    """``mcvd_oracle.make_schedule`` plus k / k_cum / theta_t for ``gamma`` configs (ncsnpp_more.py:744-749)."""
    out = O.make_schedule(config)
    if getattr(config.model, "gamma", False):
        k = out["betas"] / (out["alphas"] * (THETA_0 ** 2))
        out.update(k=k, k_cum=torch.cumsum(k.flip(0), 0).flip(0), theta_t=torch.sqrt(out["alphas"]) * THETA_0)
    return out


def noisy_cond(sched, cond: Tensor, labels: Tensor, z: Tensor) -> Tensor:
    """cond diffused to each clip's label with the NORMALISED noise z (``randn_like(cond)``, or the Gamma draw mapped
    by ``gamma_normalise``), ncsnpp_more.py:757-766.  ``alphas[labels]`` indexes the full schedule and needs integer
    labels, as in the reference."""
    used = sched["alphas"][labels].reshape(cond.shape[0], *([1] * (cond.dim() - 1)))
    return used.sqrt() * cond + (1 - used).sqrt() * z


def unet_forward(config, sd, x: Tensor, t: Tensor, cond: Tensor, cond_noise: Tensor) -> Tensor:
    """``UNetMore_DDPM.forward`` of a ``noise_in_cond`` net: noisy cond, then ``mcvd_oracle.unet_forward``."""
    return O.unet_forward(config, sd, x, t, noisy_cond(make_schedule(config), cond, t, cond_noise))


def gamma_normalise(g: Tensor, k: Tensor, theta: Tensor, alpha: Tensor) -> Tensor:
    """(g - k theta) / sqrt(1 - alpha) in fp32 as the reference writes it.  At the noisy end k theta = 1.6e5, so the
    result is quantised to fp32 ulps of g: that is the reference's noise."""
    return (g - k * theta) / (1 - alpha).sqrt()


def injected_gamma(k: Tensor, theta: Tensor, raw: Tensor) -> Tensor:
    """The Gamma 'draw' the golden generator hands the reference: g = k theta + raw sqrt(k) theta (mean and standard
    deviation of Gamma(k, scale theta)) for a standard-normal ``raw``, in fp32."""
    return k * theta + raw * k.sqrt() * theta


def cond_gamma_noise(sched, labels: Tensor, raw: Tensor) -> Tensor:
    """The normalised conditioning noise the reference derives from ``injected_gamma`` at per-clip ``labels``
    (ncsnpp_more.py:760-765: k_cum / theta_t gathered per clip and repeated to cond's shape)."""
    rep = (1,) + tuple(raw.shape[1:])
    used_k = sched["k_cum"][labels].reshape(-1, 1, 1, 1).repeat(*rep)
    used_theta = sched["theta_t"][labels].reshape(-1, 1, 1, 1).repeat(*rep)
    g = injected_gamma(used_k, used_theta, raw)
    return gamma_normalise(g, used_k, used_theta, sched["alphas"][labels].reshape(-1, 1, 1, 1))


def step_gamma_noise(sched, step: int, raw: Tensor) -> Tensor:
    """The normalised step / warm-start noise the reference's samplers derive from ``injected_gamma`` at schedule
    index ``step`` (models/__init__.py:148-151, 274-277, 319-322)."""
    k, th = sched["k_cum"][step], sched["theta_t"][step]
    return gamma_normalise(injected_gamma(k, th, raw), k, th, sched["alphas"][step])


def init_gamma(sched, raw: Tensor) -> Tensor:
    """x_T of a ``gamma`` config from ``injected_gamma``: g - k theta at index 0, NOT normalised
    (runners/ncsn_runner.py:1471-1474)."""
    k, th = sched["k_cum"][0], sched["theta_t"][0]
    return injected_gamma(k, th, raw) - k * th


@torch.no_grad()
def ddim_sample(net, sched, x: Tensor, cond=None, subsample_steps=None, denoise=True, clip_before=True, t_min=-1,
                warm_noise: Optional[Tensor] = None) -> Tensor:
    """``mcvd_oracle.ddim_sample`` plus the ``t_min`` warm start of models/__init__.py:143-153 with the normalised
    noise ``warm_noise``; final_only."""
    steps, alphas, alphas_prev, betas = O._subsample(sched, subsample_steps)
    L = len(steps)
    x_transf = False
    for i, step in enumerate(steps):
        if step < t_min * len(alphas):                                                   # :143-144
            continue
        if not x_transf and t_min > 0:                                                   # :146-153
            x = alphas[i].sqrt() * x + (1 - alphas[i]).sqrt() * warm_noise
        x_transf = True
        c_alpha, c_alpha_prev = alphas[i], alphas_prev[i]
        labels = (step * torch.ones(x.shape[0])).long()
        grad = net(x, labels, cond)
        x0 = (1 / c_alpha.sqrt()) * (x - (1 - c_alpha).sqrt() * grad)                    # :163
        if clip_before:
            x0 = x0.clip_(-1, 1)
        x = c_alpha_prev.sqrt() * x0 + (1 - c_alpha_prev).sqrt() * grad                  # :166
    if denoise:                                                                          # :194-196
        last = ((L - 1) * torch.ones(x.shape[0])).long()
        x = x - (1 - alphas[-1]).sqrt() * net(x, last, cond)
    return x.unsqueeze(0)
