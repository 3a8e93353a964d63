"""Whole-path parity on the B200 through the reference-facing API (module forward, samplers, AR loop),
against the oracle (oracle/mcvd_oracle.py, pinned to the reference) and the golden fixtures generated
from the unmodified reference (tests/golden/*.npz).

Tolerances (BASELINE.json north_star): network forward rtol 1e-3 / atol 1e-4 fp32; generated frames
PSNR >= 50 dB on [0,1] images.
"""
import numpy as np
import pytest
import torch

from common import allclose_report, golden, make_module, max_err, step_noise, write_reference_stub
from mcvd_b200 import detfill, runner, samplers
from oracle import mcvd_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RTOL, ATOL = 1e-3, 1e-4


def gpu_module(name, conv_mode="umma"):
    """conv_mode: simt | umma (round-1 tcgen05 kernel, GroupNorm partial pass) | umma+stats (same kernel, GroupNorm
    partial sums from the conv epilogue) | umma2 (CTA-pair cta_group::2 kernel, epilogue statistics)"""
    cfg, net, sd = make_module(name, DEV)
    eng = net.engine()
    eng.conv_mode = conv_mode.split("+")[0]
    eng.epilogue_stats = conv_mode in ("umma2", "umma+stats")
    return cfg, net, sd


@pytest.mark.parametrize("name", ["tiny", "tiny_spade", "tiny_rgb", "cfg1"])
@pytest.mark.parametrize("conv_mode", ["simt", "umma", "umma+stats", "umma2"])
def test_forward_parity(name, conv_mode):
    cfg, net, sd = gpu_module(name, conv_mode)
    B = cfg.bench_batch
    x, cond = detfill.synthetic_inputs(cfg, B)
    g = golden(name)
    for t in (0, 37, 990):
        tt = torch.full((B,), t, dtype=torch.long)
        mine = net(x.to(DEV), tt.to(DEV), cond=cond.to(DEV)).cpu()
        ref = torch.from_numpy(g[f"eps_t{t}"])                       # unmodified reference, CPU fp32
        bad, mx, ratio = allclose_report(mine, ref, RTOL, ATOL)
        assert bad == 0, f"{name}/{conv_mode} t={t}: {bad} elements out of tolerance, max abs err {mx:.3e}"
        orc = O.unet_forward(cfg, sd, x, tt, cond)                   # oracle restatement on this box
        bad, mx, _ = allclose_report(mine, orc, RTOL, ATOL)
        assert bad == 0, f"{name}/{conv_mode} t={t} vs oracle: max abs err {mx:.3e}"
    P = net.engine().program(B)
    assert (P.n_umma > 0) == (conv_mode != "simt")
    from mcvd_b200 import lib
    kinds = {o.kind for o in P.step_ops}
    assert (lib.OP_CONV_UMMA2 in kinds) == (conv_mode == "umma2")
    if conv_mode in ("umma2", "umma+stats") and cfg.data.image_size >= 32:
        # the GroupNorm partial pass is gone wherever the producing conv's epilogue can supply the statistics
        n_partial = sum(o.kind == lib.OP_GN_PARTIAL for o in P.step_ops)
        n_final = sum(o.kind == lib.OP_GN_FINALIZE for o in P.step_ops)
        assert n_partial < n_final // 2, (n_partial, n_final)


def test_forward_accepts_float_and_per_sample_labels():
    cfg, net, sd = gpu_module("tiny")
    B = cfg.bench_batch
    x, cond = detfill.synthetic_inputs(cfg, B)
    tt = torch.tensor([12.5, 700.0])
    mine = net(x.to(DEV), tt.to(DEV), cond=cond.to(DEV)).cpu()
    ref = O.unet_forward(cfg, sd, x, tt, cond)
    bad, mx, _ = allclose_report(mine, ref, RTOL, ATOL)
    assert bad == 0, mx


@pytest.mark.parametrize("name", ["tiny", "tiny_spade", "cfg1"])
def test_samplers_vs_reference_golden(name):
    cfg, net, sd = gpu_module(name)
    B, L = cfg.bench_batch, cfg.sampling.subsample
    x, cond = detfill.synthetic_inputs(cfg, B)
    g = golden(name)
    zs = [z.to(DEV) for z in step_noise(x.shape, L)]
    kw = dict(cond=cond.to(DEV), final_only=True, denoise=True, subsample_steps=L, clip_before=True)
    out = samplers.ddpm_sampler(x.to(DEV), net, noise_list=zs, **kw)
    assert out.shape == (1,) + tuple(x.shape) and out.is_cuda
    to01 = lambda a: ((a + 1) / 2).clamp(0, 1)
    assert O.psnr01(to01(out[0].cpu()), to01(torch.from_numpy(g["ddpm"]))) >= 50.0
    assert max_err(out[0].cpu(), torch.from_numpy(g["ddpm"])) < 5e-3
    out = samplers.ddim_sampler(x.to(DEV), net, log=False, **kw)
    assert O.psnr01(to01(out[0].cpu()), to01(torch.from_numpy(g["ddim"]))) >= 50.0
    out = samplers.FPNDM_sampler(x.to(DEV), net, cond=cond.to(DEV), final_only=True, subsample_steps=L, log=False)
    assert O.psnr01(to01(out[0].cpu()), to01(torch.from_numpy(g["fpndm"]))) >= 50.0


def test_video_gen_ar_loop_vs_golden():
    name = "tiny"
    cfg, net, sd = gpu_module(name)
    B, L = cfg.bench_batch, cfg.sampling.subsample
    x, cond = detfill.synthetic_inputs(cfg, B)
    g = golden(name)
    vid = runner.video_gen_clips(cfg, net, cond.to(DEV), cfg.sampling.num_frames_pred,
                                 init_fn=lambda i, shape: detfill.normal(f"ar_init{i}", shape).to(DEV),
                                 noise_fn=lambda i: [z.to(DEV) for z in step_noise(x.shape, L, tag=f"ar{i}_z")])
    ref = torch.from_numpy(g["video"])
    assert vid.shape == ref.shape
    assert O.psnr01(vid.cpu(), ref) >= 50.0


def test_full_size_properties_cfg2():
    """At BASELINE's headline size (cfg2: ngf 96, 64x64) the oracle is too slow for a CI loop, so check
    size-independent properties: (1) tensor-core path == CUDA-core fp32 path, (2) a clip's result does
    not depend on which batch it is in (what clip-sharding across GPUs relies on), (3) determinism."""
    cfg, net, sd = gpu_module("cfg2", "umma")
    B = 4
    x, cond = detfill.synthetic_inputs(cfg, B)
    xd, cd = x.to(DEV), cond.to(DEV)
    tt = torch.full((B,), 500, dtype=torch.long, device=DEV)
    a = net(xd, tt, cond=cd)
    a2 = net(xd, tt, cond=cd)
    assert torch.equal(a, a2), "non-deterministic"
    lo = net(xd[:2], tt[:2], cond=cd[:2])
    hi = net(xd[2:], tt[2:], cond=cd[2:])
    assert torch.equal(torch.cat([lo, hi]), a), "result depends on batch composition"
    net.engine().conv_mode = "simt"
    net.engine().programs.clear()
    b = net(xd, tt, cond=cd)
    bad, mx, _ = allclose_report(a.cpu(), b.cpu(), RTOL, ATOL)
    assert bad == 0, f"umma vs simt: max abs err {mx:.3e}"
    # one oracle evaluation of a single clip at full size anchors the magnitude
    ref = O.unet_forward(cfg, sd, x[:1], tt[:1].cpu(), cond[:1])
    bad, mx, _ = allclose_report(a[:1].cpu(), ref, RTOL, ATOL)
    assert bad == 0, f"cfg2 vs oracle: max abs err {mx:.3e}"


def test_state_dict_reload_repacks_weights():
    cfg, net, sd = gpu_module("tiny")
    B = cfg.bench_batch
    x, cond = detfill.synthetic_inputs(cfg, B)
    tt = torch.full((B,), 100, dtype=torch.long, device=DEV)
    a = net(x.to(DEV), tt, cond=cond.to(DEV)).clone()
    sd2 = {k: v.clone() for k, v in net.state_dict().items()}
    detfill.randomize_state_dict(sd2, seed=99)
    net.load_state_dict(sd2)                       # in-place parameter update, as EMAHelper.ema does
    b = net(x.to(DEV), tt, cond=cond.to(DEV))
    ref = O.unet_forward(cfg, {k: v.cpu() for k, v in sd2.items()}, x, tt.cpu(), cond)
    assert not torch.allclose(a, b)
    bad, mx, _ = allclose_report(b.cpu(), ref, RTOL, ATOL)
    assert bad == 0, mx


def test_warm_start_t_min_vs_reference_golden():
    name = "tiny_spade"
    cfg, net, sd = gpu_module(name)
    B, L = cfg.bench_batch, cfg.sampling.subsample
    x, cond = detfill.synthetic_inputs(cfg, B)
    zs = step_noise(x.shape, L)
    steps = list(range(0, 1000, 1000 // L))
    kept = [i for i, s_ in enumerate(steps) if not (s_ < 0.35 * L)]
    aligned = [None] * (L - 1)
    for k, i in enumerate(kept[:-1]):
        aligned[i] = zs[k].to(DEV)
    out = samplers.ddpm_sampler(x.to(DEV), net, cond=cond.to(DEV), final_only=True, denoise=True, subsample_steps=L,
                                clip_before=True, noise_list=aligned, t_min=0.35,
                                warm_noise=detfill.normal("warm", x.shape).to(DEV))
    g = golden(name)
    to01 = lambda a: ((a + 1) / 2).clamp(0, 1)
    assert O.psnr01(to01(out[0].cpu()), to01(torch.from_numpy(g["ddpm_tmin"]))) >= 50.0


def test_forward_parity_128px_five_levels():
    """cityscapes-like topology at 128 px: exercises 130-wide slabs (3 slab rows per producer thread), five
    resolution levels and 3-channel frames; checked against the oracle (no reference golden for this one)."""
    cfg, net, sd = gpu_module("tiny128")
    B = cfg.bench_batch
    x, cond = detfill.synthetic_inputs(cfg, B)
    tt = torch.tensor([250, 900])
    mine = net(x.to(DEV), tt.to(DEV), cond=cond.to(DEV)).cpu()
    ref = O.unet_forward(cfg, sd, x, tt, cond)
    bad, mx, _ = allclose_report(mine, ref, RTOL, ATOL)
    assert bad == 0, f"max abs err {mx:.3e}"


def test_cuda_graph_replay_is_bit_identical_to_eager_launches():
    cfg, net, sd = gpu_module("tiny")
    B, L = cfg.bench_batch, cfg.sampling.subsample
    x, cond = detfill.synthetic_inputs(cfg, B)
    kw = dict(cond=cond.to(DEV), final_only=True, denoise=True, subsample_steps=L, philox_seed=5, clip_offset=0)
    eng = net.engine()
    eng.use_graph = True
    a = samplers.ddpm_sampler(x.to(DEV), net, **kw)
    assert eng.program(B).graph is not None, "graph was not captured"
    eng.use_graph = False
    b = samplers.ddpm_sampler(x.to(DEV), net, **kw)
    assert torch.equal(a, b)


def test_samplers_accept_dataparallel_style_wrapper():
    cfg, net, sd = gpu_module("tiny")
    B, L = cfg.bench_batch, cfg.sampling.subsample
    x, cond = detfill.synthetic_inputs(cfg, B)

    class Wrapper(torch.nn.Module):          # what the reference does: scorenet = DataParallel(get_model(config))
        def __init__(self, m):
            super().__init__()
            self.module = m

        def forward(self, *a, **k):
            return self.module(*a, **k)

    kw = dict(cond=cond.to(DEV), final_only=True, subsample_steps=L, philox_seed=3)
    a = samplers.ddpm_sampler(x.to(DEV), Wrapper(net), **kw)
    b = samplers.ddpm_sampler(x.to(DEV), net, **kw)
    assert torch.equal(a, b)


@pytest.mark.parametrize("name", ["cfg3", "cfg4", "cfg5"])
def test_big_configs_forward_vs_oracle(name):
    """BASELINE.json configs[2..4] at FULL size (163 M-parameter SPADE net; ngf 192 with 192-channel heads; the 128-px
    five-level net): one clip through the CUDA path against the oracle at two timesteps, rtol 1e-3 / atol 1e-4."""
    torch.set_num_threads(min(torch.get_num_threads(), 16))
    cfg, net, sd = gpu_module(name)
    x, cond = detfill.synthetic_inputs(cfg, 1)
    for t in (37, 800):
        tt = torch.tensor([t])
        mine = net(x.to(DEV), tt.to(DEV), cond=cond.to(DEV)).cpu()
        ref = O.unet_forward(cfg, sd, x, tt, cond)
        bad, mx, ratio = allclose_report(mine, ref, RTOL, ATOL)
        assert bad == 0, f"{name} t={t}: {bad} elements out of tolerance, max abs err {mx:.3e} (x{ratio:.2f} of the limit)"
    P = net.engine().program(1)
    assert P.n_umma > 0 and P.n_simt <= 60, (P.n_umma, P.n_simt)     # only SPADE's 10-channel mlp_shared convs may be SIMT


def test_cfg2_ten_step_sampler_vs_oracle():
    """BASELINE.json configs[1] at full size: a 10-step DDPM sampler call (+ denoise) on one clip with injected
    noise against the oracle's sampler: PSNR >= 50 dB on [0,1] frames and max |diff| < 5e-3."""
    torch.set_num_threads(min(torch.get_num_threads(), 16))
    cfg, net, sd = gpu_module("cfg2")
    L = 10
    x, cond = detfill.synthetic_inputs(cfg, 1, seed=21)
    zs = step_noise(x.shape, L, tag="c2z")
    out = samplers.ddpm_sampler(x.to(DEV), net, cond=cond.to(DEV), final_only=True, denoise=True, subsample_steps=L,
                                clip_before=True, noise_list=[z.to(DEV) for z in zs])[0].cpu()
    fn = lambda xx, tt, cc: O.unet_forward(cfg, sd, xx, tt, cc)
    ref = O.ddpm_sample(fn, O.make_schedule(cfg), x.clone(), cond, L, True, True, noise=zs)[0]
    to01 = lambda a: ((a + 1) / 2).clamp(0, 1)
    assert O.psnr01(to01(out), to01(ref)) >= 50.0
    assert max_err(out, ref) < 5e-3


def test_ema_style_data_copy_triggers_repack():
    """reference EMAHelper.ema() (models/ema.py:23-28) writes through param.data.copy_(), which does NOT bump the
    parameter's version counter; the engine must still notice (value fingerprint) and repack after a forward."""
    cfg, net, sd = gpu_module("tiny")
    B = cfg.bench_batch
    x, cond = detfill.synthetic_inputs(cfg, B)
    tt = torch.full((B,), 100, dtype=torch.long, device=DEV)
    a = net(x.to(DEV), tt, cond=cond.to(DEV)).clone()          # packs weights, builds the program
    sd2 = {k: v.clone() for k, v in net.state_dict().items()}
    detfill.randomize_state_dict(sd2, seed=77)
    versions = [p._version for p in net.parameters()]
    for name_, p in net.named_parameters():
        p.data.copy_(sd2[name_].to(p.device))                   # exactly what EMAHelper.ema does
    assert versions == [p._version for p in net.parameters()]   # the hazard: counters did not move
    b = net(x.to(DEV), tt, cond=cond.to(DEV))
    ref = O.unet_forward(cfg, {k: v.cpu() for k, v in sd2.items()}, x, tt.cpu(), cond)
    assert not torch.allclose(a, b)
    bad, mx, _ = allclose_report(b.cpu(), ref, RTOL, ATOL)
    assert bad == 0, mx


def test_one_frame_at_a_time_ar_loop_vs_oracle():
    """sampling.one_frame_at_a_time (reference runners/ncsn_runner.py:1500-1501, 1534-1535): one kept frame per AR
    iteration, the conditioning window slides by one frame.  Checked against the oracle's restatement of the loop."""
    cfg, net, sd = gpu_module("tiny")
    cfg.sampling.one_frame_at_a_time = True
    nfp = 3
    B, L = cfg.bench_batch, cfg.sampling.subsample
    C, F, Fc, S = cfg.data.channels, cfg.data.num_frames, cfg.data.num_frames_cond, cfg.data.image_size
    x, cond = detfill.synthetic_inputs(cfg, B)
    shape = (B, C * F, S, S)
    inits = [detfill.normal(f"of_init{i}", shape) for i in range(nfp)]
    noises = [step_noise(shape, L, tag=f"of{i}_z") for i in range(nfp)]
    vid = runner.video_gen_clips(cfg, net, cond.to(DEV), nfp, init_fn=lambda i, sh: inits[i].to(DEV),
                                 noise_fn=lambda i: [z.to(DEV) for z in noises[i]]).cpu()
    # oracle: the same loop with the oracle sampler
    fn = lambda xx, tt, cc: O.unet_forward(cfg, sd, xx, tt, cc)
    sched = O.make_schedule(cfg)
    c, preds = cond.clone(), []
    for i in range(nfp):
        gen = O.ddpm_sample(fn, sched, inits[i].clone(), c, L, True, True, noise=noises[i])[0]
        preds.append(gen)
        c = torch.cat([c[:, C:], gen[:, :C]], dim=1)
    ref = ((torch.cat(preds, 1)[:, :C * nfp] + 1) / 2).clamp(0, 1)
    assert vid.shape == ref.shape
    assert O.psnr01(vid, ref) >= 50.0


def test_packed_weight_disk_cache(tmp_path, monkeypatch):
    """MCVD_WEIGHT_CACHE: the kernel-layout weight images are written once per checkpoint and read back by the next
    engine with the same parameter values; another checkpoint gets its own file."""
    monkeypatch.setenv("MCVD_WEIGHT_CACHE", str(tmp_path))
    cfg, net, sd = make_module("tiny", DEV)
    B = cfg.bench_batch
    x, cond = detfill.synthetic_inputs(cfg, B)
    tt = torch.full((B,), 300, dtype=torch.long, device=DEV)
    a = net(x.to(DEV), tt, cond=cond.to(DEV))
    e1 = net.engine()
    assert e1.packs_computed > 0 and e1.packs_loaded == 0
    files = list(tmp_path.glob("mcvd_b200_packed_*.pt"))
    assert len(files) == 1
    cfg2_, net2, _ = make_module("tiny", DEV)                 # same deterministic weights -> same fingerprint
    b = net2(x.to(DEV), tt, cond=cond.to(DEV))
    e2 = net2.engine()
    assert e2.packs_computed == 0 and e2.packs_loaded == e1.packs_computed
    assert torch.equal(a, b)
    sd2 = {k: v.clone() for k, v in net2.state_dict().items()}
    detfill.randomize_state_dict(sd2, seed=5)
    net2.load_state_dict(sd2)                                  # other values: a second cache file, freshly packed
    net2(x.to(DEV), tt, cond=cond.to(DEV))
    assert len(list(tmp_path.glob("mcvd_b200_packed_*.pt"))) == 2 and net2.engine().packs_computed > 0


def test_patch_install_dispatches_to_the_cuda_path(tmp_path, monkeypatch):
    """mcvd_b200.patch.install() on a CUDA box.  The reference tree is not part of this repository, so a stub with the
    reference's module layout (tests/common.py) stands in for it; with the real tree the same code path runs
    (tests/test_host_cpu.py covers the CPU fallback)."""
    import importlib
    import sys
    write_reference_stub(tmp_path)
    monkeypatch.syspath_prepend(str(tmp_path))
    for m in ("runners", "runners.ncsn_runner", "models"):
        sys.modules.pop(m, None)
    try:
        from mcvd_b200 import patch, model as fast_model
        from mcvd_b200 import configs
        patch.install(verbose=False)
        R = importlib.import_module("runners.ncsn_runner")
        M = importlib.import_module("models")
        cfg = configs.workload("tiny")
        cfg.device = torch.device(DEV)
        net = R.get_model(cfg)                                   # fast module for a covered config on CUDA
        assert isinstance(net, fast_model.UNetMore_DDPM) and next(net.parameters()).is_cuda
        sd = net.state_dict()
        detfill.randomize_state_dict(sd, 1234)
        net.load_state_dict(sd)
        x, cond = detfill.synthetic_inputs(cfg, 2)
        L = cfg.sampling.subsample
        out = M.ddpm_sampler(x.to(DEV), net, cond=cond.to(DEV), final_only=True, subsample_steps=L, philox_seed=1,
                             n_steps_each=0, step_lr=0.0, config=cfg)      # reference-only kwargs are swallowed
        assert torch.is_tensor(out) and out.shape == (1,) + tuple(x.shape) and out.is_cuda
        assert R.ddpm_sampler is M.ddpm_sampler                  # names bound by `from models import ...` follow
        cfg_cpu = configs.workload("tiny")
        cfg_cpu.device = torch.device("cpu")
        assert R.get_model(cfg_cpu) == "reference model"         # uncovered (CPU) config: the reference's own model
        assert M.ddim_sampler(x, "some reference module") == "reference ddim"
    finally:
        for m in ("runners", "runners.ncsn_runner", "models"):
            sys.modules.pop(m, None)


def test_data_parallel_replicas_build_their_own_engine():
    """torch.nn.DataParallel shallow-copies the module per device (reference runners/ncsn_runner.py:1377): a replica
    must not share the original's engine (device-0 weights, buffers and CUDA graph)."""
    cfg, net, sd = gpu_module("tiny")
    B = cfg.bench_batch
    x, cond = detfill.synthetic_inputs(cfg, B)
    tt = torch.full((B,), 10, dtype=torch.long, device=DEV)
    a = net(x.to(DEV), tt, cond=cond.to(DEV))
    assert net._engine is not None
    rep = net._replicate_for_data_parallel()
    assert rep._engine is None
    if torch.cuda.device_count() >= 2:
        dp = torch.nn.DataParallel(net, device_ids=[0, 1])
        out = dp(x.to(DEV), tt, cond=cond.to(DEV))
        assert torch.allclose(out.cpu(), a.cpu(), rtol=0, atol=0)
