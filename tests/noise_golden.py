"""Access to tests/golden/noise_options.npz (the reference with noise_in_cond / gamma, oracle/gen_noise_golden.py) for
the CPU and GPU tests.  Normal noise is the raw detfill draw itself.  Gamma noise is what the reference derived from
its injected draws: regenerated here with the oracle's restatement of the reference's fp32 expression, from the
labels and schedule indices the fixture records, and checked against the fixture's digest of every derived tensor."""
import numpy as np
import torch

from common import GOLDEN_DIR
from mcvd_b200.synthetic import make_module
from oracle import noise_oracle as N
from oracle.gen_golden import tensor_digest
from oracle.gen_noise_golden import AR_FRAMES, FWD_LABELS, noise_config, raw  # noqa: F401

_G = None


def golden():
    global _G
    if _G is None:
        _G = np.load(f"{GOLDEN_DIR}/noise_options.npz")
    return _G


def tag(name, gamma):
    return f"{name}_{'gamma' if gamma else 'normal'}"


def module(name, gamma, device):
    return make_module(noise_config(name, gamma), device)


def noise(name, gamma, key, kind, shape):
    """the normalised draws of one recorded run, in draw order: kind 'cond' (one per network call) or 'step'"""
    t, g = tag(name, gamma), golden()
    sched = N.make_schedule(noise_config(name, gamma))
    if kind == "cond":
        plan = [torch.from_numpy(lab) for lab in g[f"{t}_{key}_cond_labels"]]
        derive = lambda lab, z: N.cond_gamma_noise(sched, lab, z)
    else:
        plan = [int(s) for s in g[f"{t}_{key}_step_idx"]]
        derive = lambda s, z: N.step_gamma_noise(sched, s, z)
    zs = [raw(t, key, kind, n, shape) for n in range(len(plan))]
    if not gamma:
        return zs
    zs = [derive(p, z) for p, z in zip(plan, zs)]
    assert [tensor_digest(z) for z in zs] == list(g[f"{t}_{key}_{kind}_digest"]), (t, key, kind)
    return zs


def ar_init(name, i, shape):
    """x_T of AR iteration i of the recorded Gamma loop (the reference's g - k theta), digest-checked"""
    t = tag(name, True)
    z = N.init_gamma(N.make_schedule(noise_config(name, True)), raw(t, f"ar_init{i}", "x", 0, shape))
    assert tensor_digest(z) == golden()[f"{t}_ar_init_digest"][i]
    return z


def ref(name, gamma, key):
    return torch.from_numpy(golden()[f"{tag(name, gamma)}_{key}"])
