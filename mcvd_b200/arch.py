"""Static description of the UNetMore / NCSN++ score network derived from a config.

Mirrors the construction order of the reference (``models/better/ncsnpp_more.py:186-247`` concat
variant, ``:534-584`` SPADE variant) so that module index ``i`` here is ``unet.all_modules[i]`` there
and checkpoints load by name.  Only the 2-D, positional-embedding, BigGAN-resblock configuration the
reference hard-codes (``fir=True, skip_rescale=True, resblock_type='biggan'``, :62-66) is described;
anything else is rejected by ``check_supported``.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional


def num_groups(ch: int) -> int:
    """GroupNorm group count: min(ch // 4, 32) decremented until it divides ch (layerspp.py:474-477)."""
    g = min(ch // 4, 32)
    while ch % g != 0:
        g -= 1
    return g


@dataclass
class ModSpec:
    kind: str                      # 'linear' | 'conv3x3' | 'res' | 'attn' | 'norm'
    idx: int = -1                  # index in unet.all_modules
    in_ch: int = 0
    out_ch: int = 0
    res: int = 0                   # INPUT spatial size of the module
    up: bool = False
    down: bool = False
    skip_ch: int = 0               # channels popped from the skip stack and concatenated (up path)
    push: bool = False             # output is pushed on the skip stack
    has_shortcut: bool = False     # Conv_2 exists
    heads: int = 1
    film_off: List[int] = field(default_factory=list)   # offsets of actnorm0/1 in the fused FiLM table


@dataclass
class NetSpec:
    spade: bool
    nf: int
    temb_dim: int
    in_ch: int                     # network input channels (after the concat for the non-SPADE net)
    out_ch: int
    cond_ch: int
    image_size: int
    spade_dim: int
    n_head_channels: int
    mods: List[ModSpec]
    film_total: int                # total FiLM outputs (sum of 2*ch over every act-norm with an embedding)


def check_supported(config) -> Optional[str]:
    """Return None if the fast path covers this config, else the reason it does not."""
    m, d = config.model, config.data
    if getattr(m, "arch", None) != "unetmore":
        return f"arch={getattr(m, 'arch', None)!r} (only 'unetmore' 2-D)"
    if getattr(m, "version", "DDPM").upper() not in ("DDPM", "DDIM", "FPNDM"):
        return "version must be DDPM/DDIM/FPNDM"
    for flag in ("cond_emb", "output_all_frames"):
        if getattr(m, flag, False):
            return f"model.{flag}=True is not accelerated"
    if not getattr(m, "time_conditional", True):
        return "time_conditional=False"
    if getattr(m, "sigma_dist", "linear") != "linear":
        return "sigma_dist != linear"
    if m.ngf % 16 != 0:
        return "ngf must be a multiple of 16"
    if d.image_size % (2 ** (len(m.ch_mult) - 1)) != 0:
        return "image_size not divisible by the down-sampling factor"
    return None


def build_spec(config) -> NetSpec:
    m, d = config.model, config.data
    spade = bool(getattr(m, "spade", False))
    C, F = d.channels, d.num_frames
    Fc = d.num_frames_cond + getattr(d, "num_frames_future", 0)
    nf, ch_mult, nrb = m.ngf, list(m.ch_mult), m.num_res_blocks
    attn_res = list(m.attn_resolutions)
    nhc = m.n_head_channels
    R = len(ch_mult)
    S = d.image_size
    all_res = [S // (2 ** i) for i in range(R)]
    mods: List[ModSpec] = []
    film = [0]

    def add(ms: ModSpec):
        ms.idx = len(mods)
        mods.append(ms)
        return ms

    def heads_of(ch):
        if nhc == -1:
            return 1
        if ch < nhc:
            return 1
        assert ch % nhc == 0, f"channels {ch} not divisible by n_head_channels {nhc} (layerspp.py:227)"
        return ch // nhc

    def res(in_ch, out_ch, r, up=False, down=False, skip=0, push=False):
        tot = in_ch + skip
        ms = ModSpec("res", in_ch=tot, out_ch=out_ch, res=r, up=up, down=down, skip_ch=skip, push=push,
                     has_shortcut=(tot != out_ch or up or down))
        ms.film_off = [film[0], film[0] + 2 * tot]
        film[0] += 2 * tot + 2 * out_ch
        return add(ms)

    def attn(ch, r, push=False):
        return add(ModSpec("attn", in_ch=ch, out_ch=ch, res=r, heads=heads_of(ch), push=push))

    add(ModSpec("linear", in_ch=nf, out_ch=4 * nf))
    add(ModSpec("linear", in_ch=4 * nf, out_ch=4 * nf))
    net_in = C * F if spade else C * (F + Fc)
    add(ModSpec("conv3x3", in_ch=net_in, out_ch=nf, res=S, push=True))
    hs_c = [nf]
    in_ch = nf
    for lvl in range(R):
        r = all_res[lvl]
        for _ in range(nrb):
            out_ch = nf * ch_mult[lvl]
            has_attn = r in attn_res
            res(in_ch, out_ch, r, push=not has_attn)
            in_ch = out_ch
            if has_attn:
                attn(in_ch, r, push=True)
            hs_c.append(in_ch)
        if lvl != R - 1:
            res(in_ch, in_ch, r, down=True, push=True)
            hs_c.append(in_ch)
    r = all_res[-1]
    res(in_ch, in_ch, r)
    attn(in_ch, r)
    res(in_ch, in_ch, r)
    for lvl in reversed(range(R)):
        r = all_res[lvl]
        for _ in range(nrb + 1):
            out_ch = nf * ch_mult[lvl]
            res(in_ch, out_ch, r, skip=hs_c.pop())
            in_ch = out_ch
        if r in attn_res:
            attn(in_ch, r)
        if lvl != 0:
            res(in_ch, in_ch, r, up=True)
    assert not hs_c
    add(ModSpec("norm", in_ch=in_ch, out_ch=in_ch, res=S))
    add(ModSpec("conv3x3", in_ch=in_ch, out_ch=C * F, res=S))
    return NetSpec(spade=spade, nf=nf, temb_dim=4 * nf, in_ch=net_in, out_ch=C * F, cond_ch=C * Fc, image_size=S,
                   spade_dim=getattr(m, "spade_dim", 128), n_head_channels=nhc, mods=mods, film_total=film[0])
