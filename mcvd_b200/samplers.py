"""DDPM / DDIM / F-PNDM reverse-diffusion loops with the reference's signatures.

Drop-in for ``ddpm_sampler`` / ``ddim_sampler`` / ``FPNDM_sampler`` of the reference
``models/__init__.py:207-340, 103-203, 39-99`` (+ ``models/pndm.py``): same keyword arguments
(unknown ones are swallowed, exactly like the reference's ``**kwargs``), same return shape
``[1 or T, B, C*F, S, S]`` on the input's device.

The loop keeps the state ``x`` in a static NCHW device buffer; each step launches the lowered network
program and one fused update kernel (x0-prediction, clamp, posterior mean, + sigma * z) -- nothing is
synchronised with the host unless ``log`` / ``verbose`` ask for the reference's diagnostics.
Schedule coefficients are computed with the same fp32 torch expressions as the reference so they are
bit-identical.
"""
from __future__ import annotations

import logging
from typing import List, Optional

import numpy as np
import torch

from . import lib
from .model import UNetMore_DDPM


def _unwrap(scorenet) -> UNetMore_DDPM:
    net = scorenet.module if hasattr(scorenet, "module") else scorenet
    if not isinstance(net, UNetMore_DDPM):
        raise TypeError("mcvd_b200 samplers drive mcvd_b200.UNetMore_DDPM modules "
                        f"(got {type(net).__name__}); use the reference samplers for reference modules")
    return net


def _schedule(net, subsample_steps):
    """models/__init__.py:211-240 on CPU fp32 tensors (values identical to the reference's)."""
    alphas, alphas_prev, betas = net.alphas.detach().cpu(), net.alphas_prev.detach().cpu(), net.betas.detach().cpu()
    steps = np.arange(len(betas))
    if subsample_steps is not None and subsample_steps < len(alphas):
        skip = len(alphas) // subsample_steps
        steps = torch.tensor(list(range(0, len(alphas), skip)))
        alphas = alphas.index_select(0, steps)
        alphas_prev = torch.cat([alphas[1:], torch.tensor([1.0])])
        betas = 1.0 - torch.div(alphas, alphas_prev)
    return steps, alphas, alphas_prev, betas


def _gamma_schedule(net, steps):
    """(k_cum, theta_t) at the sampler's steps, as models/__init__.py:217-218,233-235,252-253 select them."""
    ks_cum, thetas = net.k_cum.detach().cpu(), net.theta_t.detach().cpu()
    idx = torch.as_tensor(np.asarray(steps), dtype=torch.long)
    return ks_cum[idx], thetas[idx]


def _seed(philox_seed):
    """The caller's Philox seed, or a fresh one from torch's generator (the reference draws from torch's RNG)."""
    return int(philox_seed) if philox_seed is not None else int(torch.randint(0, 2 ** 62, (1,)).item())


# Philox step keys of the draws that are not per-step noise (the per-step noise of step i uses key i)
WARM_KEY = 0x7FFFFFFE      # init_prev_t warm start
INIT_KEY = 0x7FFFFFFF      # video_gen init draw x_T


class _Loop:
    """Shared plumbing: program lookup, input staging, per-step launch."""

    def __init__(self, x_mod, scorenet, cond, cond_noise_list=None, philox=None):
        """``cond_noise_list`` / ``philox = (seed, clip0)``: conditioning noise of a ``noise_in_cond`` net, one tensor
        per network call, or drawn in-kernel keyed by (seed, clip, call ordinal); with neither, ``torch.randn`` per
        call (normal) or in-kernel under a seed from torch's generator (Gamma)."""
        self.net = _unwrap(scorenet)
        self.eng = self.net.engine()
        # the engine refuses to exist off-GPU (no CPU fallback); a CPU x_mod is staged to its device and the
        # result is returned on x_mod's device, as the reference samplers do
        self.dev = self.eng.device
        self.out_dev = x_mod.device              # results go back to the caller's device (reference contract)
        self.B = x_mod.shape[0]
        self.shape = x_mod.shape
        self.launches = 0
        if self.eng.spec.cond_ch > 0 and cond is None:
            raise RuntimeError("mcvd_b200: cond is required by this network")
        self._ctx = self.eng._devctx()
        self._ctx.__enter__()
        try:                                     # anything below may raise (build failure, OOM): do not leak the
            self.P = self.eng.program(self.B)    # current-device context
            self.eng.set_inputs(self.P, x=x_mod.to(self.dev).float(),
                                cond=None if cond is None else cond.to(self.dev).float())
            self.eng.run_cond(self.P)
            self.launches += self.P.cond_launches
            self.u = self.P.update_arr[0]
            self.calls = 0
            self.cond_noise_list = cond_noise_list
            self.cond_philox = None
            if self.P.noise_idx is not None and cond_noise_list is None and (philox is not None or self.net.gamma):
                self.cond_philox = (_seed(None if philox is None else philox[0]), 0 if philox is None else philox[1])
        except BaseException:
            self._ctx.__exit__(None, None, None)
            raise

    def close(self):
        self._ctx.__exit__(None, None, None)

    def result(self, t):
        return t.to(self.out_dev)

    def eps(self, t):
        """eps = net(x_state, t, cond) into P.eps_nhwc (x_state = P.x_in)."""
        self.eng.set_inputs(self.P, t=t)
        if self.P.noise_idx is not None:                 # noise_in_cond: this call's conditioning noise
            if self.cond_noise_list is not None:
                self.eng.set_cond_noise(self.P, z=self.cond_noise_list[self.calls].to(self.dev).float())
            elif self.cond_philox is not None:
                self.eng.set_cond_noise(self.P, philox=self.cond_philox, ordinal=self.calls)
            else:
                self.eng.set_cond_noise(self.P, z=torch.randn(self.P.cond_noise.shape, device=self.dev))
        self.calls += 1
        self.eng.run_step_graphed(self.P)
        self.launches += self.P.step_launches

    def update(self, k0, k1, ca, cb, cc, sigma, clip, noise=None, philox=None, step=0, gamma=None):
        """x = ca * x0 + cb * x + cc * eps + sigma * z.  ``gamma = (k, theta)``: z is the centred Gamma draw g - k theta
        made in-kernel under ``philox`` (sigma carries the normalisation)."""
        u = self.u
        u.f0, u.f1, u.f2, u.f3, u.f4, u.f5 = float(k0), float(k1), float(ca), float(cb), float(cc), float(sigma)
        fl = lib.F_CLIP if clip else 0
        if sigma != 0.0:
            if gamma is not None:
                seed, clip0 = philox
                fl |= lib.F_GAMMA
                u.f6, u.f7 = float(gamma[0]), float(gamma[1])
                u.i0, u.i1, u.i2, u.i3 = int(seed & 0x7FFFFFFF), int((seed >> 31) & 0x7FFFFFFF), int(clip0), int(step)
            elif philox is not None:
                seed, clip0 = philox
                fl |= lib.F_PHILOX
                u.i0, u.i1, u.i2, u.i3 = int(seed & 0x7FFFFFFF), int((seed >> 31) & 0x7FFFFFFF), int(clip0), int(step)
            else:
                self.P.noise.copy_(noise.reshape(self.P.noise.shape))
        u.flags = fl
        self.eng._run(self.P.update_arr, 1)
        self.launches += 1

    def state(self):
        return self.P.x_in.reshape(self.shape).clone()

    def eps_nchw(self):
        self.eng._run(self.P.out_arr, 1)
        self.launches += 1
        return self.P.out.reshape(self.shape)


def _warm_start(lp, c_alpha, warm_noise, gamma):
    """init_prev_t warm start, models/__init__.py:146-153 / 272-279: x = sqrt(a) x + sqrt(1 - a) z.  z = warm_noise
    when given; else normal, or with ``gamma = (k, theta, seed, clip0)`` the normalised Gamma draw made in-kernel."""
    sa, sb = c_alpha.sqrt().item(), (1 - c_alpha).sqrt().item()
    if gamma is None or warm_noise is not None:
        z0 = warm_noise if warm_noise is not None else torch.randn(lp.P.noise.shape, device=lp.dev)
        lp.update(0.0, 0.0, 0.0, sa, 0.0, sb, False, noise=z0)
    else:
        k, theta, seed, clip0 = gamma
        lp.update(0.0, 0.0, 0.0, sa, 0.0, sb / float(np.sqrt(1.0 - float(c_alpha))), False,
                  gamma=(float(k), float(theta)), philox=(seed, clip0), step=WARM_KEY)


def gamma_init(scorenet, shape, seed: int, clip_offset: int = 0) -> torch.Tensor:
    """x_T of a ``gamma`` config: g - k theta with g ~ Gamma(k_cum[0], scale theta_t[0]), NOT divided by
    sqrt(1 - alpha) (reference runners/ncsn_runner.py:1471-1474).  Drawn in-kernel by the diffusion-update op keyed by
    (seed, clip_offset + b, INIT_KEY, element), so a clip's x_T does not depend on how clips are sharded."""
    net = _unwrap(scorenet)
    eng = net.engine()
    B, C, S = shape[0], shape[1], shape[2]
    x = torch.zeros(shape, device=eng.device, dtype=torch.float32)
    eps = torch.zeros(shape, device=eng.device, dtype=torch.float32)
    if B == 0:
        return x
    op = lib.McvdOp()
    op.kind, op.B, op.H, op.W, op.C0, op.flags = lib.OP_DIFFUSION_UPDATE, B, S, shape[3], C, lib.F_GAMMA
    op.f5, op.f6, op.f7 = 1.0, float(net.k_cum[0]), float(net.theta_t[0])
    op.i0, op.i1, op.i2, op.i3 = seed & 0x7FFFFFFF, (seed >> 31) & 0x7FFFFFFF, clip_offset, INIT_KEY
    op.src0, op.dst = eps.data_ptr(), x.data_ptr()
    with eng._devctx():
        eng._run(lib.make_ops([op]), 1)
    return x


def _log_line(tag, i, L, grad, x, c_alpha, verbose, log):
    """Diagnostics of models/__init__.py:295-308 (forces host syncs, as in the reference)."""
    g = -1 / (1 - c_alpha).sqrt().item() * grad
    grad_norm = torch.norm(g.reshape(g.shape[0], -1), dim=-1).mean()
    image_norm = torch.norm(x.reshape(x.shape[0], -1), dim=-1).mean()
    grad_mean_norm = torch.norm(g.mean(dim=0).reshape(-1)) ** 2 * (1 - c_alpha).item()
    msg = "{}: {}/{}, grad_norm: {}, image_norm: {}, grad_mean_norm: {}".format(
        tag, i + 1, L, grad_norm.item(), image_norm.item(), grad_mean_norm.item())
    if verbose:
        print(msg)
    if log:
        logging.info(msg)


@torch.no_grad()
def ddpm_sampler(x_mod, scorenet, cond=None, just_beta=False, final_only=False, denoise=True, subsample_steps=None,
                 same_noise=False, noise_val=None, frac_steps=None, verbose=False, log=False, clip_before=True,
                 t_min=-1, gamma=False, noise_list: Optional[List[torch.Tensor]] = None, philox_seed=None,
                 clip_offset=0, warm_noise: Optional[torch.Tensor] = None,
                 cond_noise_list: Optional[List[torch.Tensor]] = None, **kwargs):
    """Reference ``ddpm_sampler`` (models/__init__.py:207-340).

    Extensions (keyword-only in practice): ``noise_list`` = per-step injected noise (L-1 tensors) for
    parity tests; ``philox_seed`` / ``clip_offset`` = draw the noise in-kernel from a counter-based
    stream keyed by the GLOBAL clip index, so a clip gets the same noise on any GPU.  With neither, the
    noise is ``torch.randn_like`` as in the reference (:324).

    ``gamma=True`` (:214-218, 319-322): the step noise is the normalised Gamma draw (g - k theta) / sqrt(1 - alpha),
    g ~ Gamma(k_cum[step], scale theta_t[step]), drawn in-kernel (under ``philox_seed``, else a seed from torch's
    generator); ``noise_list`` / ``warm_noise`` entries are that normalised noise.  On a ``noise_in_cond`` net
    ``cond_noise_list`` injects the conditioning noise, one tensor per network call (denoise call included).
    """
    t_min = -1 if t_min is None else t_min
    lp = _Loop(x_mod, scorenet, cond, cond_noise_list,
               None if philox_seed is None else (philox_seed, clip_offset))
    try:
        steps, alphas, alphas_prev, betas = _schedule(lp.net, subsample_steps)
        if frac_steps is not None:                                             # :249-256
            steps = steps[int((1 - frac_steps) * len(steps)):]
            alphas, alphas_prev, betas = alphas[steps], alphas_prev[steps], betas[steps]
        if gamma:
            ks_cum, thetas = _gamma_schedule(lp.net, steps)
            gseed = _seed(philox_seed)
        if same_noise and noise_val is None:                                    # :258-259
            noise_val = x_mod.detach().clone()
        L = len(steps)
        images = []
        x_transf = False
        for i, step in enumerate(steps):
            if step < t_min * len(alphas):                                      # :269-270 (init_prev_t warm start)
                continue
            if not x_transf and t_min > 0:                                      # :272-279: noise x to this level
                _warm_start(lp, alphas[i], warm_noise, (ks_cum[i], thetas[i], gseed, clip_offset) if gamma else None)
            x_transf = True
            c_beta, c_alpha, c_alpha_prev = betas[i], alphas[i], alphas_prev[i]
            lp.eps(float(step))                                                 # :283-284
            k0 = 1 / c_alpha.sqrt()                                             # :287
            k1 = (1 - c_alpha).sqrt()
            ca = c_alpha_prev.sqrt() * c_beta / (1 - c_alpha)                   # :290
            cb = (1 - c_beta).sqrt() * (1 - c_alpha_prev) / (1 - c_alpha)
            last = i + 1 == L
            sigma, noise = 0.0, None
            if not last:                                                        # :311-328
                sigma = (c_beta.sqrt() if just_beta else ((1 - c_alpha_prev) / (1 - c_alpha) * c_beta).sqrt()).item()
                if same_noise:
                    noise = noise_val
                elif noise_list is not None:
                    noise = noise_list[i]
                elif gamma:                 # in-kernel centred draw; sigma takes the 1 / sqrt(1 - alpha)
                    sigma = sigma / float(np.sqrt(1.0 - float(c_alpha)))
                elif philox_seed is None:
                    noise = torch.randn(lp.P.noise.shape, device=lp.dev, dtype=torch.float32)
            gkw = {}
            if gamma and noise is None and sigma != 0.0:
                gkw = dict(gamma=(ks_cum[i].item(), thetas[i].item()), philox=(gseed, clip_offset), step=i)
            elif sigma != 0.0:
                gkw = dict(philox=None if philox_seed is None or noise is not None else (philox_seed, clip_offset),
                           step=i)
            want_log = (verbose or log) and (i == 0 or (i + 1) % max(L // 10, 1) == 0)
            if want_log or not final_only:
                # the reference reports / stores x BEFORE the noise is added (:292-308)
                lp.update(k0.item(), k1.item(), ca.item(), cb.item(), 0.0, 0.0, clip_before)
                if not final_only:
                    images.append(lp.state().to("cpu"))
                if want_log:
                    _log_line("DDPM", i, L, lp.eps_nchw(), lp.state(), c_alpha, verbose, log)
                if sigma != 0.0:  # x += sigma * z  == update with x0-coefficient 0 and x-coefficient 1
                    lp.update(0.0, 0.0, 0.0, 1.0, 0.0, sigma, False, noise=noise, **gkw)
            else:
                lp.update(k0.item(), k1.item(), ca.item(), cb.item(), 0.0, sigma, clip_before, noise=noise, **gkw)
        if denoise:                                                             # :331-335
            lp.eps(float(L - 1))
            lp.update(0.0, 0.0, 0.0, 1.0, -(1 - alphas[-1]).sqrt().item(), 0.0, False)
            if not final_only:
                images.append(lp.state().to("cpu"))
        ddpm_sampler.last_launches = lp.launches
        if final_only:
            return lp.result(lp.state().unsqueeze(0))
        return torch.stack(images)
    finally:
        lp.close()


@torch.no_grad()
def ddim_sampler(x_mod, scorenet, cond=None, final_only=False, denoise=True, subsample_steps=None, verbose=False,
                 log=True, clip_before=True, t_min=-1, gamma=False, warm_noise: Optional[torch.Tensor] = None,
                 philox_seed=None, clip_offset=0, cond_noise_list: Optional[List[torch.Tensor]] = None, **kwargs):
    """Reference ``ddim_sampler`` (models/__init__.py:103-203): x = sqrt(a_prev) x0 + sqrt(1 - a_prev) eps.

    DDIM draws noise only for the ``t_min`` warm start (Gamma with ``gamma=True``, :146-153) and, on a
    ``noise_in_cond`` net, for the conditioning frames; ``philox_seed`` / ``clip_offset`` / ``cond_noise_list`` /
    ``warm_noise`` as in ``ddpm_sampler``."""
    t_min = -1 if t_min is None else t_min
    lp = _Loop(x_mod, scorenet, cond, cond_noise_list,
               None if philox_seed is None else (philox_seed, clip_offset))
    try:
        steps, alphas, alphas_prev, betas = _schedule(lp.net, subsample_steps)
        if gamma:
            ks_cum, thetas = _gamma_schedule(lp.net, steps)
            gseed = _seed(philox_seed)
        L = len(steps)
        images = []
        x_transf = False
        for i, step in enumerate(steps):
            if step < t_min * len(alphas):                                           # :143-144
                continue
            if not x_transf and t_min > 0:                                           # :146-153
                _warm_start(lp, alphas[i], warm_noise, (ks_cum[i], thetas[i], gseed, clip_offset) if gamma else None)
            x_transf = True
            c_alpha, c_alpha_prev = alphas[i], alphas_prev[i]
            lp.eps(float(step))
            lp.update((1 / c_alpha.sqrt()).item(), (1 - c_alpha).sqrt().item(), c_alpha_prev.sqrt().item(), 0.0,
                      (1 - c_alpha_prev).sqrt().item(), 0.0, clip_before)          # :163-166
            if not final_only:
                images.append(lp.state().to("cpu"))
            if (verbose or log) and (i == 0 or (i + 1) % max(L // 10, 1) == 0):
                _log_line("DDIM", i, L, lp.eps_nchw(), lp.state(), c_alpha, verbose, log)
        if denoise:                                                                 # :194-196
            lp.eps(float(L - 1))
            lp.update(0.0, 0.0, 0.0, 1.0, -(1 - alphas[-1]).sqrt().item(), 0.0, False)
            if not final_only:
                images.append(lp.state().to("cpu"))
        if final_only:
            return lp.result(lp.state().unsqueeze(0))
        return torch.stack(images)
    finally:
        lp.close()


@torch.no_grad()
def FPNDM_sampler(x_mod, scorenet, cond=None, final_only=False, denoise=True, subsample_steps=None, verbose=False,
                  log=True, clip_before=True, t_min=-1, gamma=False, **kwargs):
    """Reference ``FPNDM_sampler`` + ``pndm.gen_order_4`` (models/__init__.py:39-99, models/pndm.py:3-52).

    Replicated as written: alphas looked up through the flipped copy with the +1 offset, steps_next =
    [-1] + steps[:-1], fractional mid-timesteps fed to the network, no final denoise call.  Every
    network call (L + 9 of them) runs in the CUDA library; the eps history (``ets``), its 4-term linear
    combination and the per-step ``transfer`` are a handful of tiny elementwise torch ops on the GPU
    (fusing them into the update kernel is listed under "next" in DESIGN.md).
    """
    if _unwrap(scorenet).noise_in_cond and cond is not None:
        # the reference's forward indexes alphas[labels] with the fractional mid-step labels (pndm.py:42) and fails
        raise IndexError("FPNDM_sampler cannot drive a noise_in_cond network: its fractional mid-step labels cannot "
                         "index alphas (the reference raises the same IndexError)")
    lp = _Loop(x_mod, scorenet, cond)
    try:
        net = lp.net
        alphas = net.alphas.detach().cpu()
        alphas_old = alphas.flip(0)                                                  # :58
        skip = len(alphas) // subsample_steps
        steps = list(range(0, len(alphas), skip))
        steps_next = [-1] + steps[:-1]                                               # :63
        P = lp.P

        def eps_at(x, t):
            lp.eng.set_inputs(P, x=x)
            lp.eps(float(t))
            return lp.eps_nchw().clone()

        def transfer(x, t, t_next, et):
            """pndm.py:19-34.  x_next = x + (a' - a) * (cx * x - ce * et), then optional clamp."""
            at = alphas_old[int(t) + 1]
            an = alphas_old[int(t_next) + 1]
            cx = 1 / (at.sqrt() * (at.sqrt() + an.sqrt()))
            ce = 1 / (at.sqrt() * (((1 - an) * at).sqrt() + ((1 - at) * an).sqrt()))
            x_next = x + (an - at) * (cx * x - ce * et)
            return x_next.clip_(-1, 1) if clip_before else x_next

        x = x_mod.to(lp.dev).float()             # eps tensors live on the engine's device; keep x there too
        ets: List[torch.Tensor] = []
        images = []
        for i in range(len(steps)):
            t, t_next = steps[i], steps_next[i]
            t_mid = (t + t_next) / 2                                                 # pndm.py:42 (fractional)
            if len(ets) > 2:                                                         # pndm.py:44-47
                ets.append(eps_at(x, t))
                noise = (1 / 24) * (55 * ets[-1] - 59 * ets[-2] + 37 * ets[-3] - 9 * ets[-4])
            else:                                                                    # runge_kutta, pndm.py:3-17
                e1 = eps_at(x, t)
                ets.append(e1)
                # the alpha lookup truncates the fractional mid-timestep (.long(), pndm.py:20-21)
                tm_idx = int(torch.tensor(t_mid).long().item())
                x2 = transfer(x, t, tm_idx, e1)
                e2 = eps_at(x2, t_mid)
                x3 = transfer(x, t, tm_idx, e2)
                e3 = eps_at(x3, t_mid)
                x4 = transfer(x, t, t_next, e3)
                e4 = eps_at(x4, t_next)
                noise = (1 / 6) * (e1 + 2 * e2 + 2 * e3 + e4)
            x = transfer(x, t, t_next, noise)
            if not final_only:
                images.append(x.to("cpu"))
        if final_only:
            return lp.result(x.reshape(lp.shape).unsqueeze(0))
        return torch.stack(images)
    finally:
        lp.close()


def get_sampler(config):
    """Same dispatch as reference ``NCSNRunner.get_sampler`` (runners/ncsn_runner.py:2702-2714)."""
    from functools import partial
    version = getattr(config.model, "version", "DDPM").upper()
    if version == "DDPM":
        return partial(ddpm_sampler, config=config)
    if version == "DDIM":
        return partial(ddim_sampler, config=config)
    if version == "FPNDM":
        return partial(FPNDM_sampler, config=config)
    raise NotImplementedError(f"sampler for version {version!r} is not part of the accelerated path")
