"""Shared helpers for the test-suite (test infrastructure)."""
import os

import numpy as np
import torch

from mcvd_b200 import configs, detfill

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


from mcvd_b200.synthetic import make_module, allclose_report  # noqa: E402,F401


def golden(name):
    return np.load(os.path.join(GOLDEN_DIR, f"{name}.npz"))


def step_noise(shape, L, tag="z"):
    return [detfill.normal(f"{tag}{i}", shape) for i in range(L - 1)]


def max_err(a, b):
    return float((a.double() - b.double()).abs().max())


def frames_from_table(X, table):
    """Rebuild ``[B, K*C, S, S]`` from the frames of ``X [B, T, C, S, S]`` that ``table [B, K]`` names (-1: zeros);
    the inverse of ``oracle.gen_golden.frame_table``."""
    zero = torch.zeros_like(X[0, 0])
    return torch.stack([torch.cat([X[b, t] if t >= 0 else zero for t in row]) for b, row in enumerate(table)])


def write_reference_stub(root):
    """The reference's module layout (``runners.ncsn_runner.get_model``, ``models.{ddpm,ddim,FPNDM}_sampler`` -- the
    names main.py / load_model_from_ckpt.py bind, reference runners/ncsn_runner.py:180, models/__init__.py:39,103,207)
    under ``root``, with marker return values, for the tests of ``mcvd_b200.patch``."""
    (root / "runners").mkdir()
    (root / "models").mkdir()
    (root / "runners" / "__init__.py").write_text("")
    (root / "models" / "__init__.py").write_text(
        "def ddpm_sampler(x_mod, scorenet, **kw):\n    return 'reference ddpm'\n"
        "def ddim_sampler(x_mod, scorenet, **kw):\n    return 'reference ddim'\n"
        "def FPNDM_sampler(x_mod, scorenet, **kw):\n    return 'reference fpndm'\n")
    (root / "runners" / "ncsn_runner.py").write_text(
        "from models import ddpm_sampler, ddim_sampler, FPNDM_sampler\n"
        "def get_model(config):\n    return 'reference model'\n")

