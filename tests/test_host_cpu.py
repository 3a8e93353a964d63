"""CPU-side checks (-m "not gpu"): the oracle and the module against the golden vectors recorded from the
unmodified reference (oracle/gen_golden.py), the C-ABI library's exported surface, and the host logic that
does not need a GPU."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from common import frames_from_table, golden, make_module, max_err, step_noise, write_reference_stub
from mcvd_b200 import arch, configs, detfill, lib, runner
from oracle import mcvd_oracle as O
from oracle.gen_golden import tensor_digest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("name", ["tiny", "tiny_spade", "tiny_rgb", "cfg1"])
def test_oracle_matches_reference_golden_forward(name):
    cfg, net, sd = make_module(name, "cpu")
    B = cfg.bench_batch
    x, cond = detfill.synthetic_inputs(cfg, B)
    g = golden(name)
    for t in (0, 37, 990):
        out = O.unet_forward(cfg, sd, x, torch.full((B,), t, dtype=torch.long), cond)
        assert max_err(out, torch.from_numpy(g[f"eps_t{t}"])) < 2e-5


@pytest.mark.parametrize("name", ["tiny", "tiny_spade"])
def test_oracle_matches_reference_golden_samplers_and_video(name):
    cfg, net, sd = make_module(name, "cpu")
    B, L = cfg.bench_batch, cfg.sampling.subsample
    x, cond = detfill.synthetic_inputs(cfg, B)
    g = golden(name)
    sched = O.make_schedule(cfg)
    fn = lambda xx, tt, cc: O.unet_forward(cfg, sd, xx, tt, cc)
    out = O.ddpm_sample(fn, sched, x.clone(), cond, L, True, True, noise=step_noise(x.shape, L))
    assert max_err(out[0], torch.from_numpy(g["ddpm"])) < 1e-3
    out = O.ddim_sample(fn, sched, x.clone(), cond, L, True, True)
    assert max_err(out[0], torch.from_numpy(g["ddim"])) < 1e-3
    out = O.fpndm_sample(fn, sched, x.clone(), cond, L, True)
    assert max_err(out[0], torch.from_numpy(g["fpndm"])) < 1e-3
    nfp = cfg.sampling.num_frames_pred
    inits = [detfill.normal(f"ar_init{i}", x.shape) for i in range(-(-nfp // cfg.data.num_frames))]
    vid = O.video_gen_loop(cfg, lambda xT, c, i: O.ddpm_sample(fn, sched, xT.clone(), c, L, True, True,
                                                               noise=step_noise(x.shape, L, tag=f"ar{i}_z")),
                           cond, inits, nfp)
    assert O.psnr01(vid, torch.from_numpy(g["video"])) > 60.0


@pytest.mark.parametrize("name", ["tiny", "tiny_spade", "cfg1"])
def test_oracle_and_module_pinned_to_live_reference(name):
    """State-dict layout and re-randomised values of the reference's UNetMore_DDPM, and its forward at mixed
    timesteps, as recorded in tests/golden/reference_host.npz."""
    g = golden("reference_host")
    cfg, mine, sd = make_module(name, "cpu")
    keys = list(g[f"{name}_keys"])
    assert list(mine.state_dict().keys()) == keys
    assert all(tuple(v.shape) == tuple(int(d) for d in s if d >= 0)
               for v, s in zip(mine.state_dict().values(), g[f"{name}_shapes"]))
    ref_digest = dict(zip(keys, g[f"{name}_digest"]))
    assert all(tensor_digest(sd[k]) == ref_digest[k] for k in keys)
    B = cfg.bench_batch
    x, cond = detfill.synthetic_inputs(cfg, B)
    t = torch.tensor([3, 640][:B] + [77] * max(0, B - 2))
    assert max_err(O.unet_forward(cfg, sd, x, t, cond), torch.from_numpy(g[f"{name}_eps"])) < 2e-5
    # the reference's EMAHelper copies weights by parameter name into our module: every name must be one of its
    # parameters and carry the same values
    ref_params = set(g[f"{name}_params"])
    assert all(n in ref_params and tensor_digest(p) == ref_digest[n] for n, p in mine.named_parameters())


def test_library_loads_and_exports_every_declared_symbol():
    L = lib.load()
    hdr = open(os.path.join(ROOT, "include", "mcvd_b200.h")).read()
    body = hdr[hdr.index("typedef struct McvdOp"):]
    declared = set(re.findall(r"\b(mcvd_[a-z0-9_]+)\s*\(", body))
    assert declared == set(lib.EXPORTS), declared ^ set(lib.EXPORTS)
    for sym in declared:
        assert hasattr(L, sym), sym
    assert L.mcvd_abi_version() == lib.ABI_VERSION
    assert L.mcvd_sizeof_op() == ctypes.sizeof(lib.McvdOp)
    # op-kind constants of the binding == header
    for name, val in re.findall(r"(MCVD_OP_[A-Z_0-9]+)\s*=\s*(\d+)", hdr):
        py = name.replace("MCVD_", "")
        assert getattr(lib, py) == int(val), name
    for name, sh in re.findall(r"#define (MCVD_F_[A-Z_]+)\s+\(1 << (\d+)\)", hdr):
        assert getattr(lib, name.replace("MCVD_", "")) == 1 << int(sh), name


def test_validate_program_rejects_bad_ops_without_gpu():
    o = lib.McvdOp()
    o.kind, o.B = 999, 1
    with pytest.raises(RuntimeError):
        lib.validate_program(lib.make_ops([o]), 1)
    o = lib.McvdOp()
    o.kind, o.B, o.H, o.W, o.C0 = lib.OP_APPLY, 1, 4, 4, 6      # channels not a multiple of 4
    buf = torch.zeros(256)
    o.src0 = o.dst = buf.data_ptr()
    with pytest.raises(RuntimeError, match="multiples of 4"):
        lib.validate_program(lib.make_ops([o]), 1)
    # tensor-core attention needs its operand-image scratch; the size helper and the launch count are host-only
    o = lib.McvdOp()
    o.kind, o.B, o.H, o.W, o.C0, o.i0, o.i1 = lib.OP_ATTENTION_UMMA, 2, 16, 16, 192, 2, 96
    o.src0 = o.dst = buf.data_ptr()
    with pytest.raises(RuntimeError, match="scratch"):
        lib.validate_program(lib.make_ops([o]), 1)
    o.dst2 = buf.data_ptr()
    lib.validate_program(lib.make_ops([o]), 1)
    assert lib.load().mcvd_count_launches(ctypes.byref(o), 1) == 2
    assert lib.attention_scratch_bytes(2, 256, 192) == 4 * 2 * 192 * (256 + 2 * 256)
    assert lib.attention_scratch_bytes(3, 64, 32) == 4 * 3 * 32 * (128 + 2 * 64)      # Q padded to a 128-row tile


def test_product_path_fails_loudly_without_cuda():
    cfg, net, sd = make_module("tiny", "cpu")
    x, cond = detfill.synthetic_inputs(cfg, 2)
    with pytest.raises(RuntimeError, match="CUDA"):
        net(x, torch.zeros(2, dtype=torch.long), cond=cond)
    from mcvd_b200 import samplers
    with pytest.raises(RuntimeError):
        samplers.ddpm_sampler(x, net, cond=cond, subsample_steps=10)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "mcvd_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert "oracle" not in re.sub(r'""".*?"""', "", src, flags=re.S).replace("#", "\n#").split("\n#")[0] or \
                not re.search(r"^\s*(from|import)\s+oracle", src, flags=re.M), fn
            assert not re.search(r"^\s*(from|import)\s+oracle", src, flags=re.M), fn


def test_arch_spec_matches_survey_appendix_a():
    ns = arch.build_spec(configs.workload("cfg2"))
    kinds = "".join({"linear": "L", "conv3x3": "C", "res": "R", "attn": "A", "norm": "N"}[m.kind] for m in ns.mods)
    assert kinds == "LLC" + "RRR" + "RARAR" + "RARAR" + "RARA" + "RAR" + "RRRAR" + "RRRAR" + "RRRAR" + "RRR" + "NC"
    assert len(ns.mods) == 43
    assert [m.in_ch for m in ns.mods if m.kind == "res" and m.skip_ch][:4] == [768, 768, 672, 672]
    assert arch.num_groups(96) == 24 and arch.num_groups(672) == 32 and arch.num_groups(288) == 32


def test_conditioning_and_shard_helpers():
    cfg = configs.workload("tiny")
    X = torch.arange(2 * 8 * 1 * 32 * 32, dtype=torch.float32).reshape(2, 8, 1, 32, 32)
    pred, cond, mask = runner.conditioning_fn(cfg, X, num_frames_pred=5)
    assert pred.shape == (2, 5, 32, 32) and cond.shape == (2, 3, 32, 32) and mask is None
    assert torch.equal(cond, X[:, :3].reshape(2, 3, 32, 32)) and torch.equal(pred, X[:, 3:8].reshape(2, 5, 32, 32))
    g = golden("reference_host")                       # the reference's conditioning_fn on the same X
    assert torch.equal(frames_from_table(X, g["cond_arange_pred"]), pred)
    assert torch.equal(frames_from_table(X, g["cond_arange_cond"]), cond)
    covered = []
    for r in range(3):
        lo, hi = runner.shard_range(64, r, 3)
        covered += list(range(lo, hi))
    assert covered == list(range(64))
    assert runner.shard_range(4, 7, 8) == (4, 4)


@pytest.mark.parametrize("p_cond,p_fut,sync", [(0.0, 0.0, False), (0.5, 0.0, False), (0.5, 0.5, False),
                                               (0.5, 0.5, True), (0.0, 1.0, False), (0.3, 1.0, False)])
def test_conditioning_masks_match_reference_draw_for_draw(p_cond, p_fut, sync):
    """Past / future masking of the paper's "general" models (reference runner:104-147): same Bernoulli draws in
    the same order, so a seeded run returns what the reference's conditioning_fn returned (frame tables and masks
    in tests/golden/reference_host.npz)."""
    g = golden("reference_host")
    key = f"mask_{p_cond}_{p_fut}_{int(sync)}"
    cfg = configs.workload("tiny")
    cfg.data.num_frames_future = 2
    cfg.data.prob_mask_sync = sync
    n = cfg.data.num_frames_cond + cfg.data.num_frames + cfg.data.num_frames_future
    X = detfill.normal("clips", (6, n, cfg.data.channels, 32, 32))
    torch.manual_seed(7)
    p1, c1, m1 = runner.conditioning_fn(cfg, X, num_frames_pred=cfg.data.num_frames, prob_mask_cond=p_cond,
                                        prob_mask_future=p_fut)
    assert torch.equal(frames_from_table(X, g[f"{key}_pred"]), p1)
    assert torch.equal(frames_from_table(X, g[f"{key}_cond"]), c1) and c1.shape[1] == cfg.data.channels * (3 + 2)
    m0 = g[f"{key}_mask"]
    assert m1 is None if m0.size == 0 else torch.equal(torch.from_numpy(m0), m1)
    # unconditional models get every frame as the prediction target
    u1 = runner.conditioning_fn(cfg, X, conditional=False)
    assert torch.equal(frames_from_table(X, g["uncond_pred"]), u1[0]) and u1[1] is None and u1[2] is None


def test_patch_shim_installs_and_falls_back_on_cpu(tmp_path, monkeypatch):
    """mcvd_b200.patch swaps get_model / samplers inside the reference's modules (a stub of their layout, see
    tests/common.py); on a CPU config it must hand back the reference model, and the reference samplers for it."""
    import importlib
    import sys
    write_reference_stub(tmp_path)
    monkeypatch.syspath_prepend(str(tmp_path))
    for m in ("runners", "runners.ncsn_runner", "models"):
        sys.modules.pop(m, None)
    try:
        from mcvd_b200 import patch
        patch.install(verbose=False)
        R = importlib.import_module("runners.ncsn_runner")
        M = importlib.import_module("models")
        cfg = configs.workload("tiny")
        cfg.device = torch.device("cpu")
        net = R.get_model(cfg)
        assert net == "reference model"
        x, cond = detfill.synthetic_inputs(cfg, 2)
        assert M.ddpm_sampler(x, net, cond=cond, final_only=True, subsample_steps=4) == "reference ddpm"
        assert M.ddim_sampler(x, net, cond=cond) == "reference ddim"
        assert M.FPNDM_sampler(x, net, cond=cond) == "reference fpndm"
        assert R.ddpm_sampler is M.ddpm_sampler
    finally:
        for m in ("runners", "runners.ncsn_runner", "models"):
            sys.modules.pop(m, None)


def test_metrics_oracle_grey_conversion_and_ssim_properties():
    """oracle/metrics_oracle.py (checker of MCVD_OP_FRAME_METRICS): the 8-bit grey conversion equals what
    torchvision's ToPILImage + PIL's convert('RGB').convert('L') produce (reference runners/ncsn_runner.py:1590-1599),
    and the SSIM restatement has the properties of skimage's (1 on identical images, symmetric, < 1 otherwise)."""
    import numpy as np
    from oracle import metrics_oracle as M
    rng = np.random.RandomState(0)
    for C in (1, 3):
        fr = rng.rand(C, 32, 32).astype(np.float32)
        fr[0, 0, :4] = [0.0, 1.0, 0.5, 0.999]
        try:
            from PIL import Image
            u8 = (torch.from_numpy(fr).mul(255).byte()).numpy()            # torchvision ToPILImage for float tensors
            img = Image.fromarray(u8[0], mode="L") if C == 1 else Image.fromarray(np.transpose(u8, (1, 2, 0)), mode="RGB")
            want = np.asarray(img.convert("RGB").convert("L"))
            assert np.array_equal(M.to_grey_u8(fr), want)
        except ImportError:
            pass
        g = M.to_grey_u8(fr)
        assert g.dtype == np.uint8 and g.shape == (32, 32)
    a = (rng.rand(40, 40) * 255).astype(np.uint8)
    b = np.clip(a.astype(np.int32) + rng.randint(-20, 20, a.shape), 0, 255).astype(np.uint8)
    assert abs(M.ssim_u8(a, a) - 1.0) < 1e-12
    s_ab, s_ba = M.ssim_u8(a, b), M.ssim_u8(b, a)
    assert abs(s_ab - s_ba) < 1e-12 and 0.0 < s_ab < 1.0
    pf = np.zeros((6, 4, 2))
    pf[..., 0] = rng.rand(6, 4) * 0.01 + 1e-4
    pf[..., 1] = rng.rand(6, 4)
    mse, psnr, ssim = M.best_of_repeats(pf, 3)
    assert mse.shape == (2,) and np.allclose(mse[0], pf[:3, :, 0].mean(1).min())
    assert np.allclose(psnr[1], (10 * np.log10(1 / pf[3:, :, 0].mean(1))).max()) and np.allclose(ssim[0], pf[:3, :, 1].mean(1).max())
