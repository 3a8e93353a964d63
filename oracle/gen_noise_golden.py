"""Generate tests/golden/noise_options.npz from the UNMODIFIED reference.  TEST INFRASTRUCTURE.

Needs the reference tree (``MCVD_REFERENCE_ROOT``):   python -m oracle.gen_noise_golden

The reference with ``model.noise_in_cond`` (normal and Gamma noise) on the tiny / tiny_spade workloads, weights
re-randomised by ``mcvd_b200.detfill`` as in ``oracle/gen_golden.py``.  Injected draws:
  * ``torch.randn_like`` (normal conditioning and step noise; dispatched by shape because the conditioning noise of
    every forward and the per-step noise interleave) returns raw ``detfill`` normals;
  * ``torch.distributions.gamma.Gamma`` (conditioning noise, ncsnpp_more.py:762-765) and ``models.Gamma`` (the
    samplers, models/__init__.py:148-151, 274-277, 319-322) return ``noise_oracle.injected_gamma`` of raw normals.
Recorded per net: the forward at per-clip labels; on the Gamma nets DDPM, DDIM and DDIM with t_min = 0.35
(gamma=True samplers) and, on tiny, a 2-iteration AR loop; on the normal nets DDPM; the state-dict keys, shapes and
digests.  For every run, the label of each network call and the schedule index of each Gamma step draw are stored,
so the noise the reference derived regenerates from the raw draws (``noise_oracle``); a digest of every derived
Gamma tensor pins that regeneration to what the reference computed, bit for bit, without storing the noise.
"""
from __future__ import annotations

import contextlib
import os
import sys
from unittest import mock

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from mcvd_b200 import configs, detfill                          # noqa: E402
from oracle import ref_import, mcvd_oracle as O                  # noqa: E402
from oracle import noise_oracle as N                             # noqa: E402
from oracle.gen_golden import OUT, tensor_digest                 # noqa: E402

FWD_LABELS = ([0, 990], [37, 500], [999, 3])     # per-clip labels of the recorded forwards
AR_FRAMES = 4                                   # frames predicted by the recorded AR loop (2 iterations of 2)


def noise_config(name, gamma):
    cfg = configs.workload(name)
    cfg.model.noise_in_cond = True
    cfg.model.gamma = gamma
    return cfg


def raw(tag, key, kind, n, shape):
    """the n-th raw standard-normal draw of one kind ('cond' | 'step') of one recorded run"""
    return detfill.normal(f"{tag}_{key}_{kind}{n}", shape)


class _Draws:
    """Answers the reference's noise requests of one recorded run and logs what it derived."""

    def __init__(self, tag, key, sched, x_shape, cond_shape):
        self.tag, self.key, self.sched = tag, key, sched
        self.x_shape, self.cond_shape = tuple(x_shape), tuple(cond_shape)
        self.n = {"cond": 0, "step": 0}
        self.labels = None                                       # of the current forward (pre-hook)
        self.cond_labels, self.step_idx = [], []
        self.cond_digest, self.step_digest = [], []
        self.kidx = {float(v): i for i, v in enumerate(sched["k_cum"])} if "k_cum" in sched else {}

    def raw(self, kind, shape):
        z = raw(self.tag, self.key, kind, self.n[kind], shape)
        self.n[kind] += 1
        return z

    def randn_like(self, t):
        kind = "cond" if tuple(t.shape) == self.cond_shape else "step"
        assert kind == "cond" or tuple(t.shape) == self.x_shape, t.shape
        if kind == "cond":
            self.cond_labels.append(self.labels.numpy().copy())
        else:
            self.step_idx.append(-1)                             # normal noise: no schedule index involved
        return self.raw(kind, t.shape)

    def cond_gamma(self, conc, rate):
        d = self

        class G:
            def sample(self, sample_shape=torch.Size()):
                lab = d.labels
                z = d.raw("cond", conc.shape)
                rep = (1,) + tuple(conc.shape[1:])
                used_k = d.sched["k_cum"][lab].reshape(-1, 1, 1, 1).repeat(*rep)
                used_theta = d.sched["theta_t"][lab].reshape(-1, 1, 1, 1).repeat(*rep)
                assert torch.equal(used_k, conc)
                d.cond_labels.append(lab.numpy().copy())
                d.cond_digest.append(tensor_digest(N.cond_gamma_noise(d.sched, lab, z)))
                return N.injected_gamma(used_k, used_theta, z)
        return G()

    def step_gamma(self, conc, rate):
        d = self

        class G:
            def sample(self, sample_shape=torch.Size()):
                s = d.kidx[float(conc.reshape(-1)[0])]
                z = d.raw("step", tuple(sample_shape) + tuple(conc.shape))
                d.step_idx.append(s)
                d.step_digest.append(tensor_digest(N.step_gamma_noise(d.sched, s, z)))
                k, th = d.sched["k_cum"][s], d.sched["theta_t"][s]
                return N.injected_gamma(k, th, z)
        return G()

    def patch(self):
        import models as RM
        stack = contextlib.ExitStack()
        stack.enter_context(mock.patch("torch.randn_like", self.randn_like))
        stack.enter_context(mock.patch("torch.distributions.gamma.Gamma", self.cond_gamma))
        stack.enter_context(mock.patch.object(RM, "Gamma", self.step_gamma))
        return stack


def gen_noise_options():
    out = {}
    _, ddpm, ddim, _ = ref_import.ref_models()
    for name in ("tiny", "tiny_spade"):
        for gamma in (False, True):
            cfg = noise_config(name, gamma)
            net = ref_import.build_reference_net(cfg)
            tag = f"{name}_{'gamma' if gamma else 'normal'}"
            sd = net.state_dict()
            sched = N.make_schedule(cfg)
            for k in ("alphas", "k_cum", "theta_t"):
                assert k not in sd or torch.equal(sd[k], sched[k]), k
            out[f"{tag}_keys"] = np.array(list(sd))
            out[f"{tag}_shapes"] = np.array([list(v.shape) + [-1] * (4 - v.dim()) for v in sd.values()], np.int64)
            out[f"{tag}_digest"] = np.array([tensor_digest(v) for v in sd.values()], np.uint64)
            B = cfg.bench_batch
            x, cond = detfill.synthetic_inputs(cfg, B)
            L = cfg.sampling.subsample

            def record(key, fn, store=True):
                d = _Draws(tag, key, sched, x.shape, cond.shape)
                h = net.register_forward_pre_hook(lambda m, a: setattr(d, "labels", a[1]))
                try:
                    with torch.no_grad(), d.patch():
                        r = fn()
                finally:
                    h.remove()
                if store:
                    out[f"{tag}_{key}"] = r.numpy()
                out[f"{tag}_{key}_cond_labels"] = np.stack(d.cond_labels).astype(np.int64)
                out[f"{tag}_{key}_step_idx"] = np.array(d.step_idx, np.int64)
                if gamma:
                    out[f"{tag}_{key}_cond_digest"] = np.array(d.cond_digest, np.uint64)
                    out[f"{tag}_{key}_step_digest"] = np.array(d.step_digest, np.uint64)
                return r

            for j, lab in enumerate(FWD_LABELS):
                record(f"fwd{j}", lambda: net(x, torch.tensor(lab), cond=cond))
            kw = dict(cond=cond, final_only=True, denoise=True, subsample_steps=L, clip_before=True, log=False,
                      verbose=False, gamma=gamma)
            record("ddpm", lambda: ddpm(x.clone(), net, **kw)[0])
            if not gamma:
                continue
            record("ddim", lambda: ddim(x.clone(), net, **kw)[0])
            record("ddim_tmin", lambda: ddim(x.clone(), net, t_min=0.35, **kw)[0])
            if name != "tiny":
                continue
            # AR loop (runner:1501-1570, restated in the oracle); x_T of a gamma config: runners/ncsn_runner.py:1471-1474
            n_iter = -(-AR_FRAMES // cfg.data.num_frames)
            inits = [N.init_gamma(sched, raw(tag, f"ar_init{i}", "x", 0, x.shape)) for i in range(n_iter)]
            out[f"{tag}_ar_init_digest"] = np.array([tensor_digest(z) for z in inits], np.uint64)

            def sampler(x_T, c, i):
                return record(f"ar{i}", lambda: ddpm(x_T.clone(), net, **{**kw, "cond": c})[0], store=False).unsqueeze(0)
            out[f"{tag}_video"] = O.video_gen_loop(cfg, sampler, cond, inits, AR_FRAMES).numpy()
    path = os.path.join(OUT, "noise_options.npz")
    np.savez_compressed(path, **out)
    print("noise_options", os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    assert ref_import.available(), "reference tree not found"
    gen_noise_options()
