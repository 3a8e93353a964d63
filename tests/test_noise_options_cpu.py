"""noise_in_cond and Gamma diffusion noise (model.gamma) on the CPU: the oracle against the reference's outputs in
tests/golden/noise_options.npz, the module's state_dict against the reference's, the lowered programs on the op
interpreter with injected noise, and the configurations that must raise."""
import numpy as np
import pytest
import torch

import noise_golden as NG
from common import max_err
from mcvd_b200 import arch, detfill, lib, samplers, runner
from mcvd_b200.program import Engine
from op_interpreter import Interpreter
from oracle import mcvd_oracle as O
from oracle import noise_oracle as N
from oracle.gen_golden import tensor_digest

NAMES = ["tiny", "tiny_spade"]
GAMMAS = [False, True]


class NoiseInterpreter(Interpreter):
    """the interpreter plus MCVD_F_NOISE on the input-layout op (injected noise only: there is no Philox here)"""

    def exec(self, op):
        if op.kind != lib.OP_NCHW_TO_NHWC or not op.flags & lib.F_NOISE:
            return super().exec(op)
        assert not op.flags & lib.F_PHILOX, "interpreter has no Philox"
        B, H, W = op.B, op.H, op.W
        a = self.get(op.src0, B * op.C0 * H * W).view(B, op.C0, H, W)
        b = self.get(op.src1, B * op.C1 * H * W).view(B, op.C1, H, W) if op.C1 > 0 else None
        labels = self.get(op.aux0, B).long()
        alphas = self.get(op.aux1, op.i4)
        cnd = b if b is not None else a
        z = self.get(op.aux2, cnd.numel()).view(cnd.shape)
        cnd = N.noisy_cond(dict(alphas=alphas), cnd, labels, z)
        x = torch.cat([a, cnd], 1) if b is not None else cnd
        x = x.permute(0, 2, 3, 1)
        pitch = op.Cout if op.Cout > 0 else x.shape[3]
        x = torch.nn.functional.pad(x, (0, pitch - x.shape[3]))
        self.get(op.dst, x.numel()).copy_(x.reshape(-1))


def cpu_module(name, gamma, noise_in_cond=True):
    cfg = NG.noise_config(name, gamma)
    cfg.model.noise_in_cond = noise_in_cond
    cfg, net, sd = NG.make_module(cfg, "cpu")
    net._engine = Engine(net, _test_backend=NoiseInterpreter())
    return cfg, net, sd


def oracle_net(cfg, sd, cond_zs):
    it = iter(cond_zs)
    return lambda x, t, c: N.unet_forward(cfg, sd, x, t, c, next(it))


# ----------------------------------------------------------------------------- the oracle against the reference
@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("gamma", GAMMAS)
def test_oracle_matches_reference(name, gamma):
    cfg, _, sd = cpu_module(name, gamma)
    B, L = cfg.bench_batch, cfg.sampling.subsample
    x, cond = detfill.synthetic_inputs(cfg, B)
    for j, lab in enumerate(NG.FWD_LABELS):
        zc = NG.noise(name, gamma, f"fwd{j}", "cond", cond.shape)[0]
        eps = N.unet_forward(cfg, sd, x, torch.tensor(lab), cond, zc)
        assert max_err(eps, NG.ref(name, gamma, f"fwd{j}")) < 5e-5
    sched = O.make_schedule(cfg)
    zc = NG.noise(name, gamma, "ddpm", "cond", cond.shape)
    zs = NG.noise(name, gamma, "ddpm", "step", x.shape)
    out = O.ddpm_sample(oracle_net(cfg, sd, zc), sched, x.clone(), cond, L, True, True, noise=zs)[0]
    assert max_err(out, NG.ref(name, gamma, "ddpm")) < 2e-3
    if gamma:
        out = O.ddim_sample(oracle_net(cfg, sd, NG.noise(name, gamma, "ddim", "cond", cond.shape)), sched,
                            x.clone(), cond, L, True, True)[0]
        assert max_err(out, NG.ref(name, gamma, "ddim")) < 2e-3
        warm = NG.noise(name, gamma, "ddim_tmin", "step", x.shape)[0]
        out = N.ddim_sample(oracle_net(cfg, sd, NG.noise(name, gamma, "ddim_tmin", "cond", cond.shape)), sched,
                            x.clone(), cond, L, True, True, t_min=0.35, warm_noise=warm)[0]
        assert max_err(out, NG.ref(name, gamma, "ddim_tmin")) < 2e-3


def test_gamma_schedule_buffers_match_reference():
    """k / k_cum / theta_t as the module registers them equal the reference's (digests), and the oracle's copies"""
    for name in NAMES:
        cfg, net, sd = cpu_module(name, True)
        g, t = NG.golden(), NG.tag(name, True)
        assert list(sd) == list(g[f"{t}_keys"])
        assert [list(v.shape) + [-1] * (4 - v.dim()) for v in sd.values()] == g[f"{t}_shapes"].tolist()
        assert [tensor_digest(v) for v in sd.values()] == list(g[f"{t}_digest"])
        sched = N.make_schedule(cfg)
        for k in ("k", "k_cum", "theta_t"):
            assert torch.equal(sched[k], sd[k])
        # the shapes and scales of the issue: k_cum 100 .. 2.48e10, theta 6.35e-6 .. 1e-3
        assert 99.0 < float(sd["k_cum"][-1]) < 101.0 and 2.4e10 < float(sd["k_cum"][0]) < 2.5e10
        # a normal-noise noise_in_cond net has the reference's keys without the Gamma buffers
        assert list(cpu_module(name, False)[2]) == list(g[f"{NG.tag(name, False)}_keys"])


def test_check_supported():
    cfg = NG.noise_config("tiny", True)
    assert arch.check_supported(cfg) is None
    for flag in ("cond_emb", "output_all_frames"):
        c = NG.noise_config("tiny", True)
        setattr(c.model, flag, True)
        assert flag in arch.check_supported(c)


# ----------------------------------------------------------------------------- lowering on the interpreter
@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("gamma", GAMMAS)
def test_forward_lowering(name, gamma):
    cfg, net, sd = cpu_module(name, gamma)
    B = cfg.bench_batch
    x, cond = detfill.synthetic_inputs(cfg, B)
    for j, lab in enumerate(NG.FWD_LABELS):
        zc = NG.noise(name, gamma, f"fwd{j}", "cond", cond.shape)[0]
        mine = net(x, torch.tensor(lab), cond=cond, cond_noise=zc)
        assert max_err(mine, NG.ref(name, gamma, f"fwd{j}")) < 5e-5
        assert max_err(mine, N.unet_forward(cfg, sd, x, torch.tensor(lab), cond, zc)) < 5e-5
    P = net.engine().program(B)
    assert P.noise_idx == 0 and P.step_ops[0].flags & lib.F_NOISE and not P.cond_ops
    lib.validate_program(P.step_arr, len(P.step_ops))
    assert lib.load().mcvd_count_launches(P.step_arr, len(P.step_ops)) == P.step_launches


@pytest.mark.parametrize("name", NAMES)
def test_lowering_unchanged_without_noise_in_cond(name):
    """gamma alone changes no network program; noise_in_cond moves the SPADE cond ops to the head of the step
    program and adds nothing else"""
    def programs(gamma, nic):
        cfg, net, _ = cpu_module(name, gamma, noise_in_cond=nic)
        P = net.engine().program(cfg.bench_batch)
        sig = lambda ops: [(o.kind, o.flags & ~lib.F_NOISE, o.B, o.H, o.W, o.C0, o.C1, o.Cout, o.i0, o.i1, o.i2,
                            o.i3) for o in ops]
        return sig(P.cond_ops), sig(P.step_ops), P
    base_c, base_s, base = programs(False, False)
    g_c, g_s, g = programs(True, False)
    assert (g_c, g_s) == (base_c, base_s) and g.noise_idx is None
    n_c, n_s, n = programs(True, True)
    assert n_c == [] and n_s == base_c + base_s
    assert n.step_launches == base.cond_launches + base.step_launches
    assert n.temb_idx == [i + len(base_c) for i in base.temb_idx]


@pytest.mark.parametrize("name", NAMES)
def test_samplers_lowering(name):
    cfg, net, sd = cpu_module(name, True)
    B, L = cfg.bench_batch, cfg.sampling.subsample
    x, cond = detfill.synthetic_inputs(cfg, B)
    kw = dict(cond=cond, final_only=True, denoise=True, subsample_steps=L, clip_before=True, log=False, gamma=True)
    out = samplers.ddpm_sampler(x.clone(), net, noise_list=NG.noise(name, True, "ddpm", "step", x.shape),
                                cond_noise_list=NG.noise(name, True, "ddpm", "cond", cond.shape), **kw)
    assert max_err(out[0], NG.ref(name, True, "ddpm")) < 2e-3
    out = samplers.ddim_sampler(x.clone(), net, cond_noise_list=NG.noise(name, True, "ddim", "cond", cond.shape),
                                **kw)
    assert max_err(out[0], NG.ref(name, True, "ddim")) < 2e-3
    out = samplers.ddim_sampler(x.clone(), net, t_min=0.35,
                                warm_noise=NG.noise(name, True, "ddim_tmin", "step", x.shape)[0],
                                cond_noise_list=NG.noise(name, True, "ddim_tmin", "cond", cond.shape), **kw)
    assert max_err(out[0], NG.ref(name, True, "ddim_tmin")) < 2e-3
    # normal noise_in_cond net, DDPM: the reference's cond and step draws interleave; both regenerate from detfill
    cfg, net, sd = cpu_module(name, False)
    out = samplers.ddpm_sampler(x.clone(), net, noise_list=NG.noise(name, False, "ddpm", "step", x.shape),
                                cond_noise_list=NG.noise(name, False, "ddpm", "cond", cond.shape),
                                **{**kw, "gamma": False})
    assert max_err(out[0], NG.ref(name, False, "ddpm")) < 2e-3


def test_video_gen_loop_lowering():
    name = "tiny"
    cfg, net, sd = cpu_module(name, True)
    B, L = cfg.bench_batch, cfg.sampling.subsample
    x, cond = detfill.synthetic_inputs(cfg, B)
    g, t = NG.golden(), NG.tag(name, True)
    calls = []

    def sampler(x_T, scorenet, cond, **kw):
        i = len(calls)
        calls.append(i)
        return samplers.ddpm_sampler(x_T, scorenet, cond=cond, noise_list=NG.noise(name, True, f"ar{i}", "step", x.shape),
                                     cond_noise_list=NG.noise(name, True, f"ar{i}", "cond", cond.shape), **kw)
    vid = runner.video_gen_clips(cfg, net, cond, NG.AR_FRAMES, sampler=sampler,
                                 init_fn=lambda i, shape: NG.ar_init(name, i, shape))
    assert O.psnr01(vid, torch.from_numpy(g[f"{t}_video"])) > 50.0


# ----------------------------------------------------------------------------- what must raise
def test_fpndm_and_float_labels_raise():
    cfg, net, sd = cpu_module("tiny", True)
    x, cond = detfill.synthetic_inputs(cfg, cfg.bench_batch)
    with pytest.raises(IndexError):
        samplers.FPNDM_sampler(x.clone(), net, cond=cond, subsample_steps=cfg.sampling.subsample)
    assert not net.engine().programs                     # raised before anything was lowered or launched
    zc = torch.zeros_like(cond)
    with pytest.raises(IndexError):
        net(x, torch.tensor([37.0, 500.0]), cond=cond, cond_noise=zc)
    with pytest.raises(IndexError):
        net(x, torch.tensor([37, 1000]), cond=cond, cond_noise=zc)
    # without noise_in_cond, float labels stay accepted (the sinusoidal embedding takes them)
    cfg, net, _ = cpu_module("tiny", True, noise_in_cond=False)
    net(x, torch.tensor([37.0, 500.0]), cond=cond)
