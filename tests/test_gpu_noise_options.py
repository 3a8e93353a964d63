"""noise_in_cond and Gamma diffusion noise (model.gamma) on the B200: the in-kernel Gamma sampler's statistics,
parity with the reference (tests/golden/noise_options.npz) under injected noise, and clip-sharding invariance of
every in-kernel draw.  Gates as in tests/test_gpu_model.py: forward rtol 1e-3 / atol 1e-4, sampled frames
PSNR >= 50 dB and max |delta| < 5e-3."""
import importlib
import sys

import numpy as np
import pytest
import scipy.stats as st
import torch

import noise_golden as NG
from common import allclose_report, write_reference_stub
from mcvd_b200 import detfill, lib, runner, samplers
from oracle import mcvd_oracle as O
from oracle import noise_oracle as N

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RTOL, ATOL = 1e-3, 1e-4


def gamma_draws(k, theta, seed, B, clip0=0, C=4, S=256):
    """centred Gamma draws g - k theta of one DIFFUSION_UPDATE op (x = 0 + 1 * z) on a [B, C, S, S] state"""
    x = torch.zeros(B, C, S, S, device=DEV)
    eps = torch.zeros(B, S, S, C, device=DEV)
    op = lib.McvdOp()
    op.kind, op.B, op.H, op.W, op.C0, op.flags = lib.OP_DIFFUSION_UPDATE, B, S, S, C, lib.F_GAMMA
    op.f5, op.f6, op.f7 = 1.0, float(k), float(theta)
    op.i0, op.i1, op.i2, op.i3 = seed, 0, clip0, 5
    op.src0, op.dst = eps.data_ptr(), x.data_ptr()
    lib.run_program(lib.make_ops([op]), 1, torch.cuda.current_stream().cuda_stream)
    return x


@pytest.mark.parametrize("target", [100.0, 1.9e3, 1.2e7, 2.48e10])
def test_gamma_sampler_statistics(target):
    sched = N.make_schedule(NG.noise_config("tiny", True))
    s = int(torch.argmin((sched["k_cum"].double().log() - np.log(target)).abs()))
    k, theta = float(sched["k_cum"][s]), float(sched["theta_t"][s])
    a = gamma_draws(k, theta, 11, 16)
    assert a.numel() >= 4 * 1024 * 1024
    assert torch.isfinite(a).all()
    z = a.double().cpu().numpy().ravel()
    n = z / (np.sqrt(k) * theta)                                   # standardised
    se = 1.0 / np.sqrt(n.size)
    assert abs(n.mean()) < 5 * se, n.mean()
    assert abs(n.var() - 1.0) < 5 * np.sqrt(2.0) * se, n.var()
    assert abs(st.skew(n) - 2.0 / np.sqrt(k)) < 5 * np.sqrt(6.0) * se, (st.skew(n), 2.0 / np.sqrt(k))
    p = st.kstest(z, st.gamma(a=k, loc=-k * theta, scale=theta).cdf).pvalue
    assert p > 1e-3, p
    if target == 100.0:                                            # not a normal distribution in disguise
        assert st.kstest(n, "norm").pvalue < 1e-3
    assert torch.equal(a, gamma_draws(k, theta, 11, 16))           # a pure function of the key
    assert not torch.equal(a, gamma_draws(k, theta, 12, 16))
    halves = torch.cat([gamma_draws(k, theta, 11, 8, 0), gamma_draws(k, theta, 11, 8, 8)])
    assert torch.equal(a, halves)                                  # clip_offset shards draw the same noise


def gpu_module(name, gamma):
    return NG.module(name, gamma, DEV)


def frames_gate(out, ref, what):
    out, ref = out.cpu(), ref.cpu()
    to01 = lambda v: ((v + 1) / 2).clamp(0, 1)
    psnr = O.psnr01(to01(out), to01(ref))
    mx = float((out - ref).abs().max())
    assert psnr >= 50.0 and mx < 5e-3, f"{what}: PSNR {psnr:.1f} dB, max abs {mx:.2e}"


@pytest.mark.parametrize("name", ["tiny", "tiny_spade"])
@pytest.mark.parametrize("gamma", [False, True])
def test_noise_in_cond_forward_parity(name, gamma):
    cfg, net, sd = gpu_module(name, gamma)
    B = cfg.bench_batch
    x, cond = detfill.synthetic_inputs(cfg, B)
    for j, lab in enumerate(NG.FWD_LABELS):
        zc = NG.noise(name, gamma, f"fwd{j}", "cond", cond.shape)[0]
        tt = torch.tensor(lab)
        mine = net(x.to(DEV), tt.to(DEV), cond=cond.to(DEV), cond_noise=zc.to(DEV)).cpu()
        for ref, what in ((NG.ref(name, gamma, f"fwd{j}"), "golden"),
                          (N.unet_forward(cfg, sd, x, tt, cond, zc), "oracle")):
            bad, mx, _ = allclose_report(mine, ref, RTOL, ATOL)
            assert bad == 0, f"{name} gamma={gamma} labels {lab} vs {what}: max abs err {mx:.3e}"


@pytest.mark.parametrize("name", ["tiny", "tiny_spade"])
def test_gamma_samplers_parity(name):
    cfg, net, sd = gpu_module(name, True)
    B, L = cfg.bench_batch, cfg.sampling.subsample
    x, cond = detfill.synthetic_inputs(cfg, B)
    on = lambda ts: [t.to(DEV) for t in ts]
    kw = dict(cond=cond.to(DEV), final_only=True, denoise=True, subsample_steps=L, clip_before=True, log=False,
              gamma=True)
    out = samplers.ddpm_sampler(x.to(DEV), net, noise_list=on(NG.noise(name, True, "ddpm", "step", x.shape)),
                                cond_noise_list=on(NG.noise(name, True, "ddpm", "cond", cond.shape)), **kw)
    frames_gate(out[0], NG.ref(name, True, "ddpm"), "ddpm")
    out = samplers.ddim_sampler(x.to(DEV), net, cond_noise_list=on(NG.noise(name, True, "ddim", "cond", cond.shape)),
                                **kw)
    frames_gate(out[0], NG.ref(name, True, "ddim"), "ddim")
    out = samplers.ddim_sampler(x.to(DEV), net, t_min=0.35,
                                warm_noise=NG.noise(name, True, "ddim_tmin", "step", x.shape)[0].to(DEV),
                                cond_noise_list=on(NG.noise(name, True, "ddim_tmin", "cond", cond.shape)), **kw)
    frames_gate(out[0], NG.ref(name, True, "ddim_tmin"), "ddim t_min")
    # the in-kernel Gamma paths run and stay finite (per-step noise, warm start, conditioning noise)
    for fn, extra in ((samplers.ddpm_sampler, {}), (samplers.ddpm_sampler, dict(t_min=0.35)),
                      (samplers.ddim_sampler, dict(t_min=0.35))):
        o = fn(x.to(DEV), net, philox_seed=5, **kw, **extra)
        assert torch.isfinite(o).all()
        assert torch.equal(o, fn(x.to(DEV), net, philox_seed=5, **kw, **extra))
    # the normal noise_in_cond net, DDPM with interleaved cond / step draws
    cfg, net, sd = gpu_module(name, False)
    out = samplers.ddpm_sampler(x.to(DEV), net, noise_list=on(NG.noise(name, False, "ddpm", "step", x.shape)),
                                cond_noise_list=on(NG.noise(name, False, "ddpm", "cond", cond.shape)),
                                **{**kw, "gamma": False})
    frames_gate(out[0], NG.ref(name, False, "ddpm"), "ddpm normal")


@pytest.mark.parametrize("name", ["tiny", "tiny_spade"])
@pytest.mark.parametrize("gamma", [False, True])
def test_philox_cond_noise_sharding_invariance(name, gamma):
    """conditioning noise drawn in-kernel is keyed by the global clip id: two clip_offset shards == one batch"""
    cfg, net, sd = gpu_module(name, gamma)
    x, cond = detfill.synthetic_inputs(cfg, 4)
    xd, cd = x.to(DEV), cond.to(DEV)
    tt = torch.tensor([0, 37, 500, 990], device=DEV)
    eng = net.engine()
    full = eng.forward(xd, tt, cd, cond_philox=(77, 0))
    again = eng.forward(xd, tt, cd, cond_philox=(77, 0))
    lo = eng.forward(xd[:2], tt[:2], cd[:2], cond_philox=(77, 0))
    hi = eng.forward(xd[2:], tt[2:], cd[2:], cond_philox=(77, 2))
    assert torch.isfinite(full).all()
    assert torch.equal(full, again) and torch.equal(torch.cat([lo, hi]), full)
    assert not torch.equal(full, eng.forward(xd, tt, cd, cond_philox=(78, 0)))


def test_gamma_video_gen_sharded_invariance(monkeypatch):
    """Gamma x_T, Gamma step noise and Philox conditioning noise, all keyed by the global clip id: generating 3 clips
    as shards [0, 2) + [2, 3) gives exactly the single-shard result"""
    cfg, net, sd = gpu_module("tiny", True)
    _, cond = detfill.synthetic_inputs(cfg, 3)
    monkeypatch.setattr(runner, "gather_clips", lambda local, n, rank, world, group=None: local)
    kw = dict(philox_seed=99, init_seed=7, num_frames_pred=4)
    single = runner.video_gen_sharded(cfg, net, cond.to(DEV), 0, 1, **kw)
    parts = [runner.video_gen_sharded(cfg, net, cond.to(DEV), r, 2, **kw) for r in range(2)]
    assert single.shape == (3, 4 * cfg.data.channels, 32, 32) and torch.isfinite(single).all()
    assert torch.equal(torch.cat(parts), single)


def test_patch_install_dispatches_gamma_sampler(tmp_path, monkeypatch):
    write_reference_stub(tmp_path)
    monkeypatch.syspath_prepend(str(tmp_path))
    for m in ("runners", "runners.ncsn_runner", "models"):
        sys.modules.pop(m, None)
    try:
        from mcvd_b200 import patch, model as fast_model
        patch.install(verbose=False)
        R = importlib.import_module("runners.ncsn_runner")
        M = importlib.import_module("models")
        cfg = NG.noise_config("tiny", True)
        cfg.device = torch.device(DEV)
        net = R.get_model(cfg)
        assert isinstance(net, fast_model.UNetMore_DDPM) and net.gamma and net.noise_in_cond
        x, cond = detfill.synthetic_inputs(cfg, 2)
        out = M.ddpm_sampler(x.to(DEV), net, cond=cond.to(DEV), final_only=True, subsample_steps=4, gamma=True,
                             config=cfg)
        assert torch.is_tensor(out) and out.shape == (1,) + tuple(x.shape) and out.is_cuda
    finally:
        for m in ("runners", "runners.ncsn_runner", "models"):
            sys.modules.pop(m, None)
