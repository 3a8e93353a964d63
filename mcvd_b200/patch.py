"""Drop-in shim: make the UNMODIFIED reference (``main.py --config ... --video_gen``,
``load_model_from_ckpt.py``, the demo notebook) use the B200 path.

    import mcvd_b200.patch; mcvd_b200.patch.install()      # before NCSNRunner / load_model are used

``get_model`` and the three samplers are plain module attributes in the reference
(``runners/ncsn_runner.py:180`` imported from ``models``; ``load_model_from_ckpt.py`` does
``from runners.ncsn_runner import get_model`` and ``from models import ddpm_sampler, ...``), so they can
be replaced without touching the reference tree.  ``gamma`` (Gamma diffusion noise) and ``noise_in_cond`` run on
the fast path.  Configurations it does not cover (3-D archs, ``cond_emb``, ``output_all_frames``, SMLD, CPU devices)
keep the reference implementation: same results, no acceleration.  ``torch.nn.DataParallel`` wrappers are
accepted (the samplers unwrap ``.module``), but multi-GPU runs should use ``runner.video_gen_sharded``
(one process per GPU) instead of DataParallel's per-call weight broadcast.
"""
from __future__ import annotations

import functools
import sys

from . import arch


def install(verbose: bool = True):
    import torch
    import runners.ncsn_runner as R               # the reference must be importable (on sys.path)
    import models as M
    from . import model as fast_model, samplers as fast

    ref_get_model = R.get_model
    ref_samplers = {"ddpm_sampler": M.ddpm_sampler, "ddim_sampler": M.ddim_sampler, "FPNDM_sampler": M.FPNDM_sampler}

    def get_model(config):
        dev = torch.device(getattr(config, "device", "cpu"))
        why = arch.check_supported(config) if dev.type == "cuda" else "device is not CUDA"
        if why is None:
            return fast_model.get_model(config)
        if verbose:
            print(f"[mcvd_b200] falling back to the reference model: {why}", file=sys.stderr)
        return ref_get_model(config)

    def dispatch(name):
        ref_fn, fast_fn = ref_samplers[name], getattr(fast, name)

        @functools.wraps(ref_fn)
        def sampler(x_mod, scorenet, *a, **kw):
            net = scorenet.module if hasattr(scorenet, "module") else scorenet
            is_fast = isinstance(net, fast_model.UNetMore_DDPM)
            if is_fast and not x_mod.is_cuda and next(net.parameters()).device.type != "cuda":
                raise RuntimeError("mcvd_b200 module on a CPU device: the fast path is CUDA (sm_100a) only and has "
                                   "no CPU fallback; build the reference model for CPU runs")
            use_fast = is_fast
            return (fast_fn if use_fast else ref_fn)(x_mod, scorenet, *a, **kw)
        return sampler

    R.get_model = get_model
    for name in ref_samplers:
        fn = dispatch(name)
        setattr(M, name, fn)
        if hasattr(R, name):
            setattr(R, name, fn)
    for modname in ("load_model_from_ckpt",):
        mod = sys.modules.get(modname)
        if mod is not None:
            mod.get_model = get_model
            for name in ref_samplers:
                if hasattr(mod, name):
                    setattr(mod, name, getattr(M, name))
    return get_model
