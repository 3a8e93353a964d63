"""Lowering of the score network (and one reverse-diffusion step) to a C-ABI op program.

``Engine`` owns, per module instance: the packed weights (repacked lazily when a parameter's version
counter changes -- ``load_state_dict`` / ``EMAHelper.ema`` modify parameters after construction), and
one ``Program`` per batch size: statically allocated NHWC activation buffers plus three ctypes op
arrays

  * ``cond_ops``  -- everything that depends on ``cond`` only (SPADE: the 3 conv3x3 per norm that
                     produce gamma/beta, reference layerspp.py:165-168; they are independent of t and
                     x, so a sampler call runs them ONCE instead of L+1 times),
  * ``step_ops``  -- one evaluation eps = net(x, t, cond),
  * ``update_op`` -- the DDPM/DDIM update of the NCHW state, in place.

With ``noise_in_cond`` (reference ncsnpp_more.py:753-766) ``cond`` is diffused to each clip's timestep inside every
network evaluation, so nothing depends on ``cond`` alone any more: the input-layout op that reads ``cond`` carries
MCVD_F_NOISE, and on SPADE nets the cond ops move to the head of ``step_ops`` (``cond_ops`` is empty).

The walk below follows ``NCSNpp.forward`` / ``SPADE_NCSNpp.forward`` (reference
models/better/ncsnpp_more.py:251-392, 590-718) module by module.
"""
from __future__ import annotations

import contextlib
import math
import os
from typing import Dict, List, Optional, Tuple

import torch

from . import arch, lib
from .lib import McvdOp

INV_SQRT2 = float(1.0 / math.sqrt(2.0))
GN_PPC = 64          # pixels per chunk in the GroupNorm partial pass on large maps
GN_MIN_CHUNKS = 32   # ... but at least this many chunks per sample (8-pixel floor)


def gn_chunks(hw: int) -> int:
    """Chunks (CTAs per sample) of the GroupNorm partial pass: 64-pixel chunks on large maps, but never fewer
    than GN_MIN_CHUNKS chunks (8-pixel floor) so the 8x8 .. 32x32 levels still put >= 512 CTAs on the 148 SMs at B = 64
    (one chunk per sample left them latency-bound at ~22 us per launch)."""
    return max(1, min(hw // 8, max(hw // GN_PPC, GN_MIN_CHUNKS)))


class Src:
    """A (possibly virtually concatenated) NHWC activation: channels of t0 followed by channels of t1."""

    def __init__(self, t0, c0, t1=None, c1=0):
        self.t0, self.c0, self.t1, self.c1 = t0, c0, t1, c1

    @property
    def C(self):
        return self.c0 + self.c1


def _ptr(t) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _pick_nt(cout: int) -> int:
    best = 0
    for d in range(16, 257, 16):
        if cout % d == 0:
            best = d
    return best


class Program:
    def __init__(self):
        self.keep: List[torch.Tensor] = []
        self.cond_ops: List[McvdOp] = []
        self.step_ops: List[McvdOp] = []
        self.cond_arr = None
        self.step_arr = None
        self.update_arr = None
        self.n_umma = 0
        self.n_simt = 0
        self.graph = None                    # CUDA graph of step_ops (uniform-timestep variant), captured lazily
        self.temb_idx: List[int] = []        # step ops of the time-embedding MLP + fused FiLM projection
        self.film_fin_idx: List[int] = []    # GN_FINALIZE ops that read the FiLM table
        self.uniform_t = False
        self.noise_idx: Optional[int] = None  # step op that diffuses cond (noise_in_cond nets), else None

    @staticmethod
    def count_launches(ops) -> int:
        """kernel launches of an op list (the tensor-core attention op is a pre-split + the attention kernel)"""
        return sum(2 if o.kind == lib.OP_ATTENTION_UMMA else 1 for o in ops)

    @property
    def cond_launches(self) -> int:
        return self.count_launches(self.cond_ops)

    @property
    def step_launches(self) -> int:
        return self.count_launches(self.step_ops)


class Engine:
    def __init__(self, module, _test_backend=None):
        """``_test_backend`` is a seam for the CPU test-suite only (tests/op_interpreter.py executes the
        lowered program so the host logic can be checked without a GPU).  Product code never passes it:
        without it the engine requires a CUDA device and the sm_100a library, and fails loudly."""
        self.module = module
        self.spec: arch.NetSpec = module.spec
        self.device = next(module.parameters()).device
        self.backend = _test_backend
        self.lib = lib.load()
        if self.backend is None:
            if self.device.type != "cuda":
                raise RuntimeError("mcvd_b200: the module must live on a CUDA device (no CPU fallback)")
            with torch.cuda.device(self.device):
                cc = self.lib.mcvd_device_arch()
            if cc < 100:
                raise RuntimeError(f"mcvd_b200 kernels are built for sm_100a only (device reports sm_{cc}: "
                                   f"{lib.last_error()})")
        # 'umma' (single-CTA tcgen05 kernel, default) | 'umma2' (CTA-pair cta_group::2 kernel: correct, but slower on
        # this network's 96-channel layers -- DESIGN.md section 6) | 'simt' (CUDA cores)
        self.conv_mode = os.environ.get("MCVD_CONV", "umma").lower()
        self.split_mode = int(os.environ.get("MCVD_SPLIT", "3"))            # operand split (accuracy experiments)
        # GroupNorm partial sums from the conv epilogue instead of a k_gn_partial pass.  Measured on cfg2 (B200): the
        # integer statistics make the 4-warp epilogue the bottleneck of the 96-channel layers (+1.0 ms of conv time,
        # +0.5 ms in the finalize kernels) against 0.97 ms saved, so the separate pass stays the default for the
        # round-1 kernel; the CTA-pair kernel (8 epilogue warps) always uses them.
        # 1x1 skip projection (Conv_2): 'auto' runs it on the input-stationary 1x1 kernel (conv1x1_umma.cu) and adds
        # the result as the residual of Conv_1 when that kernel takes it (<= 320 input channels), else rides along
        # Conv_1 as a second K-segment; '1' always fuses (round-1 behaviour), '0' never
        self.fuse_shortcut = os.environ.get("MCVD_FUSE_SC", "auto")
        self.epilogue_stats = os.environ.get("MCVD_EPISTATS", "1" if self.conv_mode == "umma2" else "0") == "1"
        self.attn_mode = os.environ.get("MCVD_ATTN", "umma").lower()        # 'umma' | 'simt'
        self.use_graph = os.environ.get("MCVD_GRAPH", "1") != "0"
        self.packed: Dict[str, object] = {}
        self.packed_version = None
        # optional on-disk cache of the packed (kernel-layout fp16 hi/lo) conv weights, keyed by a fingerprint of the
        # checkpoint: MCVD_WEIGHT_CACHE=<dir> (SURVEY.md section 8f row 4).  Packing a 163 M-parameter checkpoint takes
        # ~0.3 s of GPU time plus one program build; the cache turns it into a file read.
        self.cache_dir = os.environ.get("MCVD_WEIGHT_CACHE") or None
        self.packs_computed = 0
        self.packs_loaded = 0
        self.programs: Dict[int, Program] = {}
        self.launches_last_forward = 0

    # ------------------------------------------------------------------------------ weights
    MAX_PROGRAMS = 3                 # lowered programs (one per batch size) kept alive; least recently used goes first

    def _version(self):
        """Fingerprint of the parameter VALUES.  ``Tensor._version`` is not enough: the reference's
        ``EMAHelper.ema`` (models/ema.py:23-28) writes through ``param.data.copy_``, and ``.data`` carries its own
        version counter, so the parameter's stays put.  Two multi-tensor norm launches (L2 and L1 of every
        parameter, ~0.1 ms for 50 M parameters) and one comparison on the device; called once per sampler call /
        module forward, never inside the step loop."""
        ps = [p.detach() for p in self.module.parameters()]
        ids = tuple((p.data_ptr(), tuple(p.shape)) for p in ps)
        with torch.no_grad():
            fp = torch.stack(list(torch._foreach_norm(ps, 2)) + list(torch._foreach_norm(ps, 1))).double()
        return ids, fp

    def invalidate(self):
        """Forget packed weights, lowered programs and captured graphs (call after changing parameters in a way
        the fingerprint cannot see, e.g. permuting values inside one tensor)."""
        self.packed_version = None

    def _sd(self, key):
        return self._params[key]

    # -- packed-weight disk cache -----------------------------------------------------------------------
    def _cache_path(self):
        if not self.cache_dir or self.backend is not None or self.packed_version is None:
            return None
        import hashlib
        ids, fp = self.packed_version
        h = hashlib.sha256()
        h.update(repr((lib.ABI_VERSION, self.conv_mode, self.split_mode, [sh for _, sh in ids])).encode())
        h.update(fp.detach().cpu().numpy().tobytes())
        return os.path.join(self.cache_dir, f"mcvd_b200_packed_{h.hexdigest()[:32]}.pt")

    def _load_weight_cache(self):
        path = self._cache_path()
        if path is None or not os.path.exists(path):
            return
        try:
            blob = torch.load(path, map_location=self.device)
        except Exception:
            return                                       # unreadable cache: pack again
        for k, (t, scale) in blob.items():
            self.packed[k] = (t.to(self.device), scale)
            self._cache_loaded_keys.add(k)
        self.packs_loaded += len(blob)

    def _save_weight_cache(self):
        path = self._cache_path()
        if path is None:
            return
        blob = {k: (v[0].cpu(), v[1]) for k, v in self.packed.items()
                if isinstance(k, tuple) and len(k) > 1 and k[1] in ("umma", "umma2")}
        if not blob or set(blob) <= self._cache_loaded_keys:
            return                                       # nothing new since the cache was read
        os.makedirs(self.cache_dir, exist_ok=True)
        tmp = f"{path}.tmp{os.getpid()}"
        torch.save(blob, tmp)
        os.replace(tmp, path)
        self._cache_loaded_keys = set(blob)

    def ensure_packed(self):
        v = self._version()
        if self.packed_version is not None and self.packed_version[0] == v[0] and \
                torch.equal(self.packed_version[1], v[1]):
            return
        self._params = {k: p.detach() for k, p in self.module.named_parameters()}
        self.packed = {}
        self.programs = {}          # programs hold pointers into the packed tensors
        self.packed_version = v
        self._cache_loaded_keys = set()
        self._load_weight_cache()
        ns = self.spec
        # timestep-embedding frequencies, exactly as the reference computes them (layers.py:508-511)
        half = ns.nf // 2
        e = math.log(10000) / (half - 1)
        self.packed["freqs"] = torch.exp(torch.arange(half, dtype=torch.float32) * -e).to(self.device)
        # fused FiLM projection: every Dense_0 of every act-norm stacked into one [film_total, 4nf] matrix
        ws, bs = [], []
        for ms in ns.mods:
            if ms.kind == "res":
                for an in ("actnorm0", "actnorm1"):
                    ws.append(self._sd(f"unet.all_modules.{ms.idx}.{an}.Dense_0.weight"))
                    bs.append(self._sd(f"unet.all_modules.{ms.idx}.{an}.Dense_0.bias"))
        self.packed["film_w"] = torch.cat(ws, 0).contiguous().float()
        self.packed["film_b"] = torch.cat(bs, 0).contiguous().float()
        assert self.packed["film_w"].shape[0] == ns.film_total

    def _conv_taps(self, w: torch.Tensor) -> torch.Tensor:
        """OIHW -> [taps][I][O] fp32 contiguous."""
        O, I, kh, kw = w.shape
        return w.permute(2, 3, 1, 0).reshape(kh * kw, I, O).contiguous().float()

    def _pack_simt(self, taps: torch.Tensor) -> Tuple[torch.Tensor, int]:
        T, I, O = taps.shape
        OP = (O + 3) // 4 * 4
        if OP != O:
            p = torch.zeros(T, I, OP, device=taps.device, dtype=torch.float32)
            p[:, :, :O] = taps
            taps = p
        return taps.contiguous(), OP

    def _devctx(self):
        return torch.cuda.device(self.device) if self.device.type == "cuda" else contextlib.nullcontext()

    def _pack_umma(self, taps: torch.Tensor, nt: int, kb: int):
        if self.backend is not None:
            return self.backend.pack_umma(taps, nt, kb)
        self.packs_computed += 1
        T, I, O = taps.shape
        amax = float(taps.abs().max().item())
        k = 0 if amax == 0.0 else int(math.floor(math.log2(512.0 / amax)))
        k = max(-24, min(24, k))
        out = torch.empty(T * I * O * 4, device=taps.device, dtype=torch.uint8)
        stream = self._stream()
        with self._devctx():
            rc = self.lib.mcvd_umma_pack_weights(taps.data_ptr(), T, I, O, nt, kb, out.data_ptr(), k, stream)
        if rc < 0:
            raise RuntimeError(f"mcvd_b200 umma_pack_weights failed: {lib.last_error()}")
        return out, float(2.0 ** (-k))

    def _pack_umma_fused(self, taps: torch.Tensor, taps_sc: torch.Tensor, nt: int, kb: int):
        """main conv + 1x1 shortcut as one weight stream: per n-tile [main stages | shortcut stages]."""
        if self.backend is not None:
            both = torch.cat([taps.reshape(-1), taps_sc.reshape(-1)]).contiguous()
            t, _ = self.backend.pack_umma(both, nt, kb)
            return t, 1.0
        self.packs_computed += 1
        amax = float(max(taps.abs().max().item(), taps_sc.abs().max().item()))
        k = 0 if amax == 0.0 else int(math.floor(math.log2(512.0 / amax)))
        k = max(-24, min(24, k))
        n_nt = taps.shape[2] // nt
        parts = []
        for t in (taps, taps_sc):
            T, I, O = t.shape
            out = torch.empty(T * I * O * 4, device=t.device, dtype=torch.uint8)
            with self._devctx():
                rc = self.lib.mcvd_umma_pack_weights(t.data_ptr(), T, I, O, nt, kb, out.data_ptr(), k, self._stream())
            if rc < 0:
                raise RuntimeError(f"mcvd_b200 umma_pack_weights failed: {lib.last_error()}")
            parts.append(out.view(n_nt, -1))
        return torch.cat(parts, dim=1).contiguous().view(-1), float(2.0 ** (-k))

    def _pack_umma2(self, taps: torch.Tensor, taps_sc: Optional[torch.Tensor], nt: int, kb: int):
        """CTA-pair weight images (conv_umma2.cu): main conv stages, then the fused 1x1 shortcut's, per n tile."""
        if self.backend is not None:
            flat = taps.reshape(-1) if taps_sc is None else torch.cat([taps.reshape(-1), taps_sc.reshape(-1)])
            t, _ = self.backend.pack_umma(flat.contiguous(), nt, kb)
            return t, 1.0
        self.packs_computed += 1
        amax = float(taps.abs().max().item())
        if taps_sc is not None:
            amax = max(amax, float(taps_sc.abs().max().item()))
        k = 0 if amax == 0.0 else int(math.floor(math.log2(512.0 / amax)))
        k = max(-24, min(24, k))
        T, I, O = taps.shape
        isc = 0 if taps_sc is None else taps_sc.shape[1]
        per_unit = (I // kb) * T + isc // kb
        out = torch.empty((T * I + isc) * O * 4, device=taps.device, dtype=torch.uint8)
        with self._devctx():
            rc = self.lib.mcvd_umma2_pack_weights(taps.data_ptr(), T, I, O, nt, kb, out.data_ptr(), k, 0, per_unit,
                                                  self._stream())
            if rc >= 0 and taps_sc is not None:
                rc = self.lib.mcvd_umma2_pack_weights(taps_sc.data_ptr(), 1, isc, O, nt, kb, out.data_ptr(), k,
                                                      (I // kb) * T, per_unit, self._stream())
        if rc < 0:
            raise RuntimeError(f"mcvd_b200 umma2_pack_weights failed: {lib.last_error()}")
        return out, float(2.0 ** (-k))

    # ------------------------------------------------------------------------------ lowering
    def program(self, B: int, check_weights: bool = True) -> Program:
        """The lowered program for batch size B.  Every program owns its activation buffers (a few GB at the
        BASELINE batch sizes), so only MAX_PROGRAMS are kept: uneven shards / last batches evict the least
        recently used one instead of piling up."""
        if B <= 0:
            raise ValueError(f"mcvd_b200: batch size {B} (an empty shard?) cannot be lowered")
        if check_weights or self.packed_version is None:
            self.ensure_packed()
        if B in self.programs:
            self.programs[B] = self.programs.pop(B)            # most recently used last
            return self.programs[B]
        while len(self.programs) >= self.MAX_PROGRAMS:
            old = next(iter(self.programs))
            del self.programs[old]
            if self.device.type == "cuda":
                torch.cuda.empty_cache()
        with self._devctx():
            self.programs[B] = self._build(B)
            self._save_weight_cache()
        if self.backend is not None:
            self._register_all(self.programs[B])
        return self.programs[B]

    def _register_all(self, P):
        def reg(v):
            if isinstance(v, torch.Tensor):
                self.backend.register(v)
            elif isinstance(v, (tuple, list)):
                for e in v:
                    reg(e)
        for t in P.keep:
            reg(t)
        for v in self.packed.values():
            reg(v)

    def _build(self, B: int) -> Program:
        ns = self.spec
        dev = self.device
        P = Program()
        P.B = B
        S = ns.image_size

        def f32(*shape):
            t = torch.empty(shape, device=dev, dtype=torch.float32)
            P.keep.append(t)
            return t

        def keep(t):
            P.keep.append(t)
            return t

        def emit(ops, kind, **kw):
            o = McvdOp()
            o.kind = kind
            o.B = B
            for k, v in kw.items():
                if k in ("src0", "src1", "w", "bias", "aux0", "aux1", "aux2", "dst", "dst2", "src2", "src3"):
                    if isinstance(v, torch.Tensor):
                        v = v.data_ptr()
                    setattr(o, k, v)
                else:
                    setattr(o, k, v)
            ops.append(o)
            return o

        sd = self._sd
        step, cnd = P.step_ops, P.cond_ops

        # ---- convolution (tensor-core or CUDA-core) -------------------------------------------
        def conv(ops, key, src: Src, H: int, cout: int, ks: int, wname: str, bname: str, residual=None,
                 scale=1.0, tab=None, act_in=False, act_out=False, nin=False, wcat=None, bcat=None, shortcut=None,
                 stats=False):
            """dst = scale * (conv(act(norm(src))) + bias + residual [+ conv1x1(shortcut src)]).
            stats: the output feeds a GroupNorm -- let the conv epilogue emit its partial sums."""
            if wcat is not None:
                taps, bias = wcat, bcat
            elif nin:
                taps = sd(wname).float().unsqueeze(0).contiguous()          # NIN W[in, out] == [1][I][O]
                bias = sd(bname).float().contiguous()
            else:
                taps = self._conv_taps(sd(wname))
                bias = sd(bname).float().contiguous()
            keep(bias)
            dst = f32(B, H, H, cout)
            nt = _pick_nt(cout) if cout % 16 == 0 else 0
            if self.conv_mode == "umma2" and nt:
                nt = lib.umma2_pick_nt(cout, ks)
                sc_src = sc_taps = None
                c2 = c3 = 0
                if shortcut is not None:
                    sc_src, sc_w, sc_b = shortcut
                    c2, c3 = sc_src.c0, sc_src.c1
                pimg = (H + 1) * (H + 1) if ks == 3 else H * H
                want_stats = bool(stats and pimg >= 64)
                kb = lib.umma2_plan(H, H, ks, src.c0, src.c1, c2, c3, nt, want_stats)
                if kb:
                    if shortcut is not None:
                        sc_taps = self._conv_taps(sd(sc_w))
                        bias = keep((bias + sd(sc_b).float()).contiguous())
                    pk = (key, "umma2", nt, kb, shortcut is not None)
                    if pk not in self.packed:
                        self.packed[pk] = self._pack_umma2(taps, sc_taps, nt, kb)
                    wp, wscale = self.packed[pk]
                    fl = (lib.F_ACT_IN if act_in else 0) | (lib.F_ACT_OUT if act_out else 0)
                    kw2 = {}
                    if shortcut is not None:
                        kw2 = dict(src2=sc_src.t0, src3=sc_src.t1, C2=c2, C3=c3)
                    st = None
                    if want_stats:
                        st = keep(torch.zeros(lib.umma2_stats_bytes(B, H, H, ks, cout) // 8, device=dev,
                                              dtype=torch.int64))
                        stats_of[dst.data_ptr()] = (st, ks)
                    emit(ops, lib.OP_CONV_UMMA2, H=H, W=H, C0=src.c0, C1=src.c1, Cout=cout, i0=ks, i1=nt, i2=kb,
                         i3=self.split_mode, f0=scale, f1=wscale, src0=src.t0, src1=src.t1, w=wp, bias=bias,
                         aux0=residual, aux1=None if tab is None else tab3_of[tab.data_ptr()], dst=dst, dst2=st,
                         flags=fl, **kw2)
                    P.n_umma += 1
                    return dst
                nt = _pick_nt(cout)
            kb = lib.umma_kblock(src.c0, src.c1) if self.conv_mode == "umma" else 0
            sc = None
            if shortcut is not None:                       # (Src, wname, bname): 1x1 Conv_2 of the skip branch
                sc_src, sc_w, sc_b = shortcut
                kb2 = lib.umma_kblock(sc_src.c0, sc_src.c1) if kb else 0
                k1_ok = kb2 == 32 and sc_src.C <= 320 and lib.conv1x1_enabled()
                fuse = self.fuse_shortcut == "1" or (self.fuse_shortcut == "auto" and not k1_ok)
                if kb and nt and kb2 and (tab is None or H >= 8) and fuse:
                    kb = min(kb, kb2)
                    sc = (sc_src, self._conv_taps(sd(sc_w)))
                    bias = keep((bias + sd(sc_b).float()).contiguous())
                else:                                       # not fusable: separate 1x1 conv, added as residual
                    assert residual is None
                    residual = conv(ops, key + ".sc", sc_src, H, cout, 1, sc_w, sc_b)
            if kb and nt and (tab is None or H >= 8):      # fused-norm slab stages <= 8 images' table rows
                pk = (key, "umma", nt, kb, sc is not None)
                if pk not in self.packed:
                    if sc is None:
                        self.packed[pk] = self._pack_umma(taps, nt, kb)
                    else:                                  # both segments share one power-of-two scale
                        self.packed[pk] = self._pack_umma_fused(taps, sc[1], nt, kb)
                wp, wscale = self.packed[pk]
                nacc = 0                       # auto: chosen by the launcher (TMEM double-buffering, grid fill)
                fl = (lib.F_ACT_IN if act_in else 0) | (lib.F_ACT_OUT if act_out else 0)
                kw2 = {}
                if sc is not None:
                    kw2 = dict(src2=sc[0].t0, src3=sc[0].t1, C2=sc[0].c0, C3=sc[0].c1)
                st = None
                pimg = (H + 1) * (H + 1) if ks == 3 else H * H
                if stats and pimg >= 64 and self.epilogue_stats:   # GroupNorm partial sums from the epilogue
                    st = keep(torch.zeros(lib.umma2_stats_bytes(B, H, H, ks, cout) // 8, device=dev, dtype=torch.int64))
                    stats_of[dst.data_ptr()] = (st, ks)
                emit(ops, lib.OP_CONV_UMMA, H=H, W=H, C0=src.c0, C1=src.c1, Cout=cout, i0=ks, i1=nt, i2=nacc,
                     i3=self.split_mode, f0=scale, f1=wscale, src0=src.t0, src1=src.t1, w=wp, bias=bias, aux0=residual, aux1=tab,
                     dst=dst, dst2=st, flags=fl, **kw2)
                P.n_umma += 1
                return dst
            if tab is not None:
                a = f32(B, H, H, src.C)
                emit(ops, lib.OP_APPLY, H=H, W=H, C0=src.c0, C1=src.c1, src0=src.t0, src1=src.t1, aux0=tab, dst=a,
                     flags=lib.F_ACT_OUT if act_in else 0)
                src = Src(a, src.C)
            pk = (key, "simt")
            if pk not in self.packed:
                self.packed[pk] = self._pack_simt(taps)
            wp, coutp = self.packed[pk]
            emit(ops, lib.OP_CONV_SIMT, H=H, W=H, C0=src.c0, C1=src.c1, Cout=cout, i0=ks, i1=coutp, f0=scale,
                 src0=src.t0, src1=src.t1, w=wp, bias=bias, aux0=residual, dst=dst,
                 flags=lib.F_ACT_OUT if act_out else 0)
            P.n_simt += 1
            return dst

        # ---- GroupNorm statistics -> (mean, rstd, G, S) table -----------------------------------
        part_cache: Dict[int, torch.Tensor] = {}

        def partials_of(ops, t: torch.Tensor, C: int, H: int, nchunk: int):
            """per-channel (sum, sum of squares) of one tensor, computed ONCE however many norms read it"""
            key = t.data_ptr()
            if key not in part_cache:
                part = torch.empty(B * nchunk * C * 2, device=dev, dtype=torch.float64)
                keep(part)
                emit(ops, lib.OP_GN_PARTIAL, H=H, W=H, C0=C, i0=nchunk, src0=t, dst=part)
                part_cache[key] = part
            return part_cache[key]

        stats_of: Dict[int, Tuple[torch.Tensor, int]] = {}     # tensor -> (conv-epilogue tile statistics, conv ks)
        tab3_of: Dict[int, torch.Tensor] = {}                   # float4 table -> planar table (CONV_UMMA2 reads it)

        def stat_source(ops, t: torch.Tensor, C: int, H: int, nchunk: int):
            """(array, kind): the producing conv's epilogue statistics (kind = its kernel size) when it wrote
            them, else the chunk partials of a separate pass over the tensor (kind 0)"""
            if t.data_ptr() in stats_of:
                return stats_of[t.data_ptr()]
            return partials_of(ops, t, C, H, nchunk), 0

        def norm_table(ops, src: Src, H: int, eps: float, film_off=None, affine=None):
            C = src.C
            cg = C // arch.num_groups(C)
            nchunk = gn_chunks(H * H)
            tab = f32(B, C, 4)
            p0, k0 = stat_source(ops, src.t0, src.c0, H, nchunk)
            p1, k1 = stat_source(ops, src.t1, src.c1, H, nchunk) if src.t1 is not None else (None, 0)
            kw = dict(H=H, W=H, C0=src.c0, C1=src.c1, i0=nchunk, i1=cg, f0=eps, src0=p0, src1=p1, dst=tab, i4=k0,
                      i5=k1)
            if self.conv_mode == "umma2":
                tab3_of[tab.data_ptr()] = f32(B, 3, C)
                kw["dst2"] = tab3_of[tab.data_ptr()]
            if film_off is not None:
                kw.update(aux0=P.film, i2=ns.film_total, i3=film_off, flags=lib.F_FILM)
                if ops is step:
                    P.film_fin_idx.append(len(ops))
            elif affine is not None:
                kw.update(aux0=keep(affine[0].float().contiguous()), aux1=keep(affine[1].float().contiguous()))
            emit(ops, lib.OP_GN_FINALIZE, **kw)
            return tab

        # ---- SPADE gamma / beta (cond-only; reference layerspp.py:165-168) -------------------------
        cond_at: Dict[int, torch.Tensor] = {}

        def cond_resized(H):
            if H not in cond_at:
                if H == S:
                    cond_at[H] = P.cond_nhwc
                else:
                    t = f32(B, H, H, ns.cond_ch)
                    emit(cnd, lib.OP_RESIZE_NEAREST, H=H, W=H, C0=ns.cond_ch, i0=S, i1=S, src0=P.cond_nhwc, dst=t)
                    cond_at[H] = t
            return cond_at[H]

        def spade_gb(prefix: str, C: int, H: int):
            seg = cond_resized(H)
            a = conv(cnd, prefix + "mlp_shared", Src(seg, ns.cond_ch), H, ns.spade_dim, 3,
                     prefix + "mlp_shared.0.weight", prefix + "mlp_shared.0.bias", act_out=True)
            g = conv(cnd, prefix + "mlp_gamma", Src(a, ns.spade_dim), H, C, 3, prefix + "mlp_gamma.weight",
                     prefix + "mlp_gamma.bias")
            b = conv(cnd, prefix + "mlp_beta", Src(a, ns.spade_dim), H, C, 3, prefix + "mlp_beta.weight",
                     prefix + "mlp_beta.bias")
            return g, b

        # ---- inputs ---------------------------------------------------------------------------------
        P.x_in = f32(B, ns.out_ch, S, S)
        P.cond_in = f32(B, ns.cond_ch, S, S) if ns.cond_ch > 0 else None
        P.t = f32(B)
        P.out = f32(B, ns.out_ch, S, S)
        # skinny first / last convs: zero-pad K (input channels) / N (output channels) to 16 so they run on the
        # tensor-core kernel instead of the CUDA-core ones
        tc_edges = self.conv_mode in ("umma", "umma2")
        in_pad = (ns.in_ch + 15) // 16 * 16 if tc_edges else ns.in_ch
        out_pad = (ns.out_ch + 15) // 16 * 16 if tc_edges else ns.out_ch
        P.noise = f32(B, ns.out_ch, S, S)
        noisy = bool(self.module.noise_in_cond) and ns.cond_ch > 0
        nkw = {}
        if noisy:
            # cond = sqrt(a[t_b]) cond + sqrt(1 - a[t_b]) z: labels are the timestep input P.t; z is P.cond_noise until
            # set_cond_noise switches the op to in-kernel Philox (control block P.noise_ctl in device memory)
            m = self.module
            T = m.alphas.numel()
            tabs = [m.alphas] + ([m.k_cum, m.theta_t] if m.gamma else [torch.zeros_like(m.alphas)] * 2)
            P.sched_tab = keep(torch.cat([t.detach().float().reshape(-1) for t in tabs]).to(dev).contiguous())
            P.cond_noise = f32(B, ns.cond_ch, S, S)
            P.noise_ctl = keep(torch.zeros(4, device=dev, dtype=torch.int32))
            nkw = dict(flags=lib.F_NOISE, aux0=P.t, aux1=P.sched_tab, aux2=P.cond_noise, w=P.noise_ctl, i4=T)
        if ns.spade:
            P.cond_nhwc = f32(B, S, S, ns.cond_ch)
            emit(cnd, lib.OP_NCHW_TO_NHWC, H=S, W=S, C0=ns.cond_ch, src0=P.cond_in, dst=P.cond_nhwc, **nkw)
            xin = f32(B, S, S, in_pad)
            emit(step, lib.OP_NCHW_TO_NHWC, H=S, W=S, C0=ns.out_ch, Cout=in_pad, src0=P.x_in, dst=xin)
        else:
            xin = f32(B, S, S, in_pad)
            emit(step, lib.OP_NCHW_TO_NHWC, H=S, W=S, C0=ns.out_ch, C1=ns.cond_ch, Cout=in_pad, src0=P.x_in,
                 src1=P.cond_in, dst=xin, **nkw)

        # ---- time embedding + all FiLM projections (ncsnpp_more.py:273-280; layerspp.py:521) --------
        mods = ns.mods
        emb, h0, temb = f32(B, ns.nf), f32(B, ns.temb_dim), f32(B, ns.temb_dim)
        P.film = f32(B, ns.film_total)
        P.temb_idx = list(range(len(step), len(step) + 4))
        emit(step, lib.OP_TIMESTEP_EMBED, Cout=ns.nf, src0=P.t, w=self.packed["freqs"], dst=emb)
        emit(step, lib.OP_LINEAR, C0=ns.nf, Cout=ns.temb_dim, src0=emb, w=keep(sd("unet.all_modules.0.weight").float().contiguous()),
             bias=keep(sd("unet.all_modules.0.bias").float().contiguous()), dst=h0, flags=lib.F_ACT_OUT)
        emit(step, lib.OP_LINEAR, C0=ns.temb_dim, Cout=ns.temb_dim, src0=h0,
             w=keep(sd("unet.all_modules.1.weight").float().contiguous()),
             bias=keep(sd("unet.all_modules.1.bias").float().contiguous()), dst=temb, flags=lib.F_ACT_OUT)
        emit(step, lib.OP_LINEAR, C0=ns.temb_dim, Cout=ns.film_total, src0=temb, w=self.packed["film_w"],
             bias=self.packed["film_b"], dst=P.film)

        # ---- blocks ---------------------------------------------------------------------------------
        def resblock(ms: arch.ModSpec, src: Src) -> torch.Tensor:
            pre = f"unet.all_modules.{ms.idx}."
            Hin = ms.res
            H = Hin * 2 if ms.up else (Hin // 2 if ms.down else Hin)
            Cin, Cout = ms.in_ch, ms.out_ch
            eps = 1e-6 if ns.spade else 1e-5           # MySPADE param-free GN eps (layerspp.py:131) vs get_norm (:477)
            tab0 = norm_table(step, src, Hin, eps, film_off=ms.film_off[0])
            resample = lib.F_UP if ms.up else (lib.F_DOWN if ms.down else 0)
            sc_src = src
            if ns.spade or resample:
                g0 = b0 = None
                if ns.spade:
                    g0, b0 = spade_gb(pre + "actnorm0.Norm_0.", Cin, Hin)
                a0 = f32(B, H, H, Cin)
                xs = f32(B, H, H, Cin) if resample else None   # FIR of the skip branch too (layerspp.py:600-611)
                emit(step, lib.OP_APPLY, H=H, W=H, C0=src.c0, C1=src.c1, src0=src.t0, src1=src.t1, aux0=tab0, aux1=g0,
                     aux2=b0, dst=a0, dst2=xs, flags=lib.F_ACT_OUT | resample)
                if resample:
                    sc_src = Src(xs, Cin)
                h = conv(step, pre + "Conv_0", Src(a0, Cin), H, Cout, 3, pre + "Conv_0.weight", pre + "Conv_0.bias",
                         stats=True)
            else:
                h = conv(step, pre + "Conv_0", src, H, Cout, 3, pre + "Conv_0.weight", pre + "Conv_0.bias", tab=tab0,
                         act_in=True, stats=True)
            tab1 = norm_table(step, Src(h, Cout), H, eps, film_off=ms.film_off[1])
            shortcut = res = None
            if ms.has_shortcut:                      # Conv_2 rides along Conv_1 as a second K-segment
                shortcut = (sc_src, pre + "Conv_2.weight", pre + "Conv_2.bias")
            else:
                assert src.t1 is None and src.c0 == Cout
                res = src.t0
            if ns.spade:
                g1, b1 = spade_gb(pre + "actnorm1.Norm_0.", Cout, H)
                a1 = f32(B, H, H, Cout)
                emit(step, lib.OP_APPLY, H=H, W=H, C0=Cout, src0=h, aux0=tab1, aux1=g1, aux2=b1, dst=a1,
                     flags=lib.F_ACT_OUT)
                return conv(step, pre + "Conv_1", Src(a1, Cout), H, Cout, 3, pre + "Conv_1.weight",
                            pre + "Conv_1.bias", residual=res, scale=INV_SQRT2, shortcut=shortcut, stats=True)
            return conv(step, pre + "Conv_1", Src(h, Cout), H, Cout, 3, pre + "Conv_1.weight", pre + "Conv_1.bias",
                        residual=res, scale=INV_SQRT2, tab=tab1, act_in=True, shortcut=shortcut, stats=True)

        attn_scratch = [None]

        def attnblock(ms: arch.ModSpec, x: torch.Tensor) -> torch.Tensor:
            pre = f"unet.all_modules.{ms.idx}."
            H, C = ms.res, ms.in_ch
            tab = norm_table(step, Src(x, C), H, 1e-6,
                             affine=(sd(pre + "GroupNorm_0.weight"), sd(pre + "GroupNorm_0.bias")))
            wq = torch.cat([sd(pre + f"NIN_{i}.W").float() for i in range(3)], dim=1).unsqueeze(0).contiguous()
            bq = torch.cat([sd(pre + f"NIN_{i}.b").float() for i in range(3)], dim=0).contiguous()
            qkv = conv(step, pre + "qkv", Src(x, C), H, 3 * C, 1, None, None, tab=tab, act_in=False, wcat=wq, bcat=bq)
            att = f32(B, H, H, C)
            d = C // ms.heads
            T = H * H
            kt = min(T, 128 if d <= 96 else (64 if d <= 128 else 32))
            use_tc = self.attn_mode == "umma" and d in (32, 48, 64, 96, 128, 192) and T % kt == 0 and kt in (32, 64, 128)
            if use_tc:
                # q/k/v operand images (fp16 hi/lo); one scratch serves every attention layer (stream order)
                need = lib.attention_scratch_bytes(B, T, C)
                if attn_scratch[0] is None or attn_scratch[0].numel() < need:
                    attn_scratch[0] = keep(torch.empty(need, device=dev, dtype=torch.uint8))
                emit(step, lib.OP_ATTENTION_UMMA, H=H, W=H, C0=C, i0=ms.heads, i1=d, f0=float(int(d) ** (-0.5)),
                     src0=qkv, dst=att, dst2=attn_scratch[0])
            else:
                emit(step, lib.OP_ATTENTION, H=H, W=H, C0=C, i0=ms.heads, i1=d, f0=float(int(d) ** (-0.5)),
                     src0=qkv, dst=att)
            return conv(step, pre + "NIN_3", Src(att, C), H, C, 1, pre + "NIN_3.W", pre + "NIN_3.b", residual=x,
                        scale=INV_SQRT2, nin=True, stats=True)

        w_first = self._conv_taps(sd("unet.all_modules.2.weight"))
        if in_pad != ns.in_ch:
            wp_ = torch.zeros(9, in_pad, ns.nf, device=dev, dtype=torch.float32)
            wp_[:, :ns.in_ch] = w_first
            w_first = wp_
        h = conv(step, "first", Src(xin, in_pad), S, ns.nf, 3, None, None, wcat=w_first,
                 bcat=sd("unet.all_modules.2.bias").float().contiguous(), stats=True)
        hs: List[Tuple[torch.Tensor, int]] = [(h, ns.nf)]
        cur, cur_c = h, ns.nf
        for ms in mods[3:-2]:
            if ms.kind == "res":
                if ms.skip_ch:
                    st, sc = hs.pop()
                    assert sc == ms.skip_ch and cur_c + sc == ms.in_ch
                    src = Src(cur, cur_c, st, sc)
                else:
                    assert cur_c == ms.in_ch
                    src = Src(cur, cur_c)
                cur, cur_c = resblock(ms, src), ms.out_ch
            elif ms.kind == "attn":
                cur = attnblock(ms, cur)
            else:
                raise AssertionError(ms.kind)
            if ms.push:
                hs.append((cur, cur_c))
        assert not hs, "skip stack not empty"

        # ---- final norm + conv (ncsnpp_more.py:375-379) ----------------------------------------------
        mn, mc = mods[-2], mods[-1]
        pre = f"unet.all_modules.{mn.idx}."
        wl = self._conv_taps(sd(f"unet.all_modules.{mc.idx}.weight"))
        bl = keep(sd(f"unet.all_modules.{mc.idx}.bias").float().contiguous())
        pk = ("last", "simt")
        if pk not in self.packed:
            self.packed[pk] = self._pack_simt(wl)
        wlp, coutp = self.packed[pk]
        if ns.spade:
            tabn = norm_table(step, Src(cur, cur_c), S, 1e-6)
            gN, bN = spade_gb(pre + "Norm_0.", cur_c, S)
            an = f32(B, S, S, cur_c)
            emit(step, lib.OP_APPLY, H=S, W=S, C0=cur_c, src0=cur, aux0=tabn, aux1=gN, aux2=bN, dst=an,
                 flags=lib.F_ACT_OUT)
            last_src, tabn = an, None
        else:
            tabn = norm_table(step, Src(cur, cur_c), S, 1e-5,
                              affine=(sd(pre + "Norm_0.weight"), sd(pre + "Norm_0.bias")))
            last_src = cur
        if tc_edges:
            wl_p = torch.zeros(9, cur_c, out_pad, device=dev, dtype=torch.float32)
            wl_p[:, :, :ns.out_ch] = wl
            bl_p = torch.zeros(out_pad, device=dev, dtype=torch.float32)
            bl_p[:ns.out_ch] = bl
            P.eps_nhwc = conv(step, "last", Src(last_src, cur_c), S, out_pad, 3, None, None, tab=tabn, act_in=True,
                              wcat=wl_p, bcat=bl_p)
        elif ns.out_ch <= 16 and coutp * 9 * cur_c * 4 <= 200 * 1024:
            P.eps_nhwc = f32(B, S, S, ns.out_ch)
            emit(step, lib.OP_CONV_SMALLN, H=S, W=S, C0=cur_c, Cout=ns.out_ch, i1=coutp, src0=last_src, w=wlp, bias=bl,
                 aux0=tabn, dst=P.eps_nhwc, flags=lib.F_ACT_OUT)
        else:
            P.eps_nhwc = f32(B, S, S, ns.out_ch)
            if tabn is not None:
                an = f32(B, S, S, cur_c)
                emit(step, lib.OP_APPLY, H=S, W=S, C0=cur_c, src0=cur, aux0=tabn, dst=an, flags=lib.F_ACT_OUT)
                last_src = an
            emit(step, lib.OP_CONV_SIMT, H=S, W=S, C0=cur_c, Cout=ns.out_ch, i0=3, i1=coutp, f0=1.0, src0=last_src,
                 w=wlp, bias=bl, dst=P.eps_nhwc)
        P.eps_nhwc.zero_()           # read (times 0) by the warm-start noising update before the first network call
        if noisy:
            P.noise_idx = 0
            if cnd:                  # SPADE: the cond program now depends on t and runs in every evaluation
                n = len(cnd)
                step[:0] = cnd
                del cnd[:]
                P.temb_idx = [i + n for i in P.temb_idx]
                P.film_fin_idx = [i + n for i in P.film_fin_idx]
            assert step[P.noise_idx].flags & lib.F_NOISE
        P.n_net_ops = len(step)

        P.cond_arr = lib.make_ops(cnd) if cnd else None
        P.step_arr = lib.make_ops(step)
        # eps NHWC -> NCHW for the module-level forward()
        o = McvdOp()
        o.kind, o.B, o.H, o.W, o.C0 = lib.OP_NHWC_TO_NCHW, B, S, S, ns.out_ch
        o.C1 = out_pad
        o.src0, o.dst = P.eps_nhwc.data_ptr(), P.out.data_ptr()
        P.out_arr = lib.make_ops([o])
        # reverse-diffusion update (coefficients patched per step by the sampler)
        u = McvdOp()
        u.kind, u.B, u.H, u.W, u.C0 = lib.OP_DIFFUSION_UPDATE, B, S, S, ns.out_ch
        u.Cout = out_pad
        u.src0, u.src1, u.dst = P.eps_nhwc.data_ptr(), P.noise.data_ptr(), P.x_in.data_ptr()
        P.update_arr = lib.make_ops([u])
        lib.validate_program(P.step_arr, len(step))
        if cnd:
            lib.validate_program(P.cond_arr, len(cnd))
        return P

    # ------------------------------------------------------------------------------ execution
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream if self.device.type == "cuda" else 0

    def _run(self, arr, n):
        if self.backend is not None:
            self.backend.run(arr, n)
        else:
            lib.run_program(arr, n, self._stream())

    def run_cond(self, P: Program):
        if P.cond_arr is not None:
            self._run(P.cond_arr, len(P.cond_ops))

    def run_step(self, P: Program):
        self._run(P.step_arr, len(P.step_ops))

    def run_step_graphed(self, P: Program):
        """One network evaluation replayed from a CUDA graph (the ~260 launches of a forward are captured once
        per program; the timestep lives in device memory, so one graph serves every step).  Only the
        uniform-timestep variant is captured -- that is what every sampler step uses."""
        if self.backend is not None or not self.use_graph or not P.uniform_t:
            return self.run_step(P)
        if P.graph is None:
            torch.cuda.synchronize(self.device)
            g = torch.cuda.CUDAGraph()
            self.run_step(P)                                   # warm (module loading, func attributes) outside capture
            with torch.cuda.graph(g):
                self.run_step(P)
            P.graph = g
        P.graph.replay()

    def set_uniform_t(self, P: Program, uniform: bool):
        """All clips share one timestep (every sampler step): evaluate the time-embedding MLP and the fused
        FiLM projection for ONE row and let every GN_FINALIZE read it with batch stride 0 -- B x fewer
        FLOPs and bytes for the [B, 4nf] x [4nf, film_total] projection."""
        if P.uniform_t == uniform:
            return
        for i in P.temb_idx:
            P.step_arr[i].B = 1 if uniform else P.B
        for i in P.film_fin_idx:
            P.step_arr[i].i2 = 0 if uniform else self.spec.film_total
        P.uniform_t = uniform
        P.graph = None                 # kernel arguments changed: a captured graph would replay stale ones

    def set_cond_noise(self, P: Program, philox=None, ordinal: int = 0, z=None):
        """Noise source of the next evaluations of a ``noise_in_cond`` program.  ``philox = (seed, clip0)``: drawn
        in-kernel (normal, or normalised Gamma on a ``gamma`` net) keyed by (seed, clip0 + b, ordinal, element); the
        key lives in device memory, so a captured graph stays valid.  Otherwise z comes from ``P.cond_noise``
        (``z`` is copied there when given)."""
        op = P.step_arr[P.noise_idx]
        fl = lib.F_NOISE
        if philox is not None:
            fl |= lib.F_PHILOX | (lib.F_GAMMA if self.module.gamma else 0)
            seed, clip0 = philox
            key = [seed & 0x7FFFFFFF, (seed >> 31) & 0x7FFFFFFF, clip0]
            if getattr(P, "noise_key", None) != key:          # once per sampler call: a host-to-device copy
                P.noise_ctl[:3].copy_(torch.tensor(key, dtype=torch.int32))
                P.noise_key = key
            P.noise_ctl[3:].fill_(ordinal)                    # every call: one small kernel, no host synchronisation
        elif z is not None:
            P.cond_noise.copy_(z.reshape(P.cond_noise.shape))
        if op.flags != fl:
            op.flags = fl
            P.graph = None             # kernel arguments changed: a captured graph would replay stale ones

    def set_inputs(self, P: Program, x=None, t=None, cond=None):
        if x is not None:
            P.x_in.copy_(x.reshape(P.x_in.shape))
        if t is not None:
            if torch.is_tensor(t):
                self.set_uniform_t(P, False)
                P.t.copy_(t.reshape(-1).to(torch.float32))
            else:
                self.set_uniform_t(P, True)
                P.t.fill_(float(t))
        if cond is not None and P.cond_in is not None:
            P.cond_in.copy_(cond.reshape(P.cond_in.shape))

    def forward(self, x, y, cond=None, cond_noise=None, cond_philox=None):
        """One network evaluation with the reference's NCHW interface.  On a ``noise_in_cond`` net the conditioning
        noise is ``cond_noise`` (a tensor shaped like cond) or, with ``cond_philox = (seed, clip0)``, drawn
        in-kernel."""
        ns = self.spec
        B = x.shape[0]
        if ns.cond_ch > 0 and cond is None:
            raise RuntimeError("mcvd_b200: this network was built with conditioning frames; cond is required")
        with self._devctx():
            P = self.program(B)
            self.set_inputs(P, x.float(), y, cond.float() if cond is not None else None)
            if P.noise_idx is not None:
                self.set_cond_noise(P, philox=cond_philox, z=None if cond_noise is None else cond_noise.float())
            self.run_cond(P)
            self.run_step(P)
            self._run(P.out_arr, 1)
            self.launches_last_forward = P.cond_launches + P.step_launches + 1
            return P.out.clone()
