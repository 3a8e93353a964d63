/*
 * mcvd_b200 -- C ABI of the B200-native MCVD DDPM-sampling hot path.
 *
 * Plain C: device pointers and sizes only, no torch types.  Every pointer is a BORROWED device
 * pointer (owned by the caller, normally a torch tensor); outputs and workspaces are caller
 * allocated; every launch goes to the cudaStream_t passed in; no call synchronises.
 * Return value: 0 on success, negative on error (text via mcvd_last_error()).
 *
 * What this replaces in the reference (voletiv/mcvd-pytorch @ 451da2e, paths relative to its root):
 *   - the only native surface the reference has is the pybind11 op
 *       upfirdn2d(Tensor input, Tensor kernel, int up_x, up_y, down_x, down_y, pad_x0, pad_x1, pad_y0, pad_y1)
 *     (models/better/op/upfirdn2d.cpp:11-22, upfirdn2d_kernel.cu:209-369) -> MCVD_OP_APPLY with
 *     MCVD_F_UP / MCVD_F_DOWN (the FIR is fused with the norm/activation that precedes it);
 *   - everything else on the path is ATen/cuDNN/cuBLAS reached from Python
 *     (models/better/layerspp.py, layers.py, ncsnpp_more.py, models/__init__.py); the op kinds below
 *     are the fused B200 equivalents, each citing the reference lines it stands for.
 *
 * The host side (mcvd_b200/program.py) lowers a network + sampler step into an array of McvdOp and
 * calls mcvd_run_program() once per network evaluation (or once per CUDA-graph capture).
 */
#ifndef MCVD_B200_H
#define MCVD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MCVD_ABI_VERSION 5

/* ---- op kinds ------------------------------------------------------------------------------- */
enum {
  /* [B,C0,H,W] (+ [B,C1,H,W]) fp32 NCHW -> [B,H,W,C0+C1] NHWC.  torch.cat([x, cond], 1) +
   * x.contiguous() of ncsnpp_more.py:256-257,293.  Cout > 0: destination channel pitch (extra channels
   * are zero-filled so the first conv can run on the tensor cores with K a multiple of 16).
   * MCVD_F_NOISE: the conditioning frames (src1 when C1 > 0, else src0) are diffused to each clip's timestep on the
   * way, UNetMore_DDPM.forward with noise_in_cond (ncsnpp_more.py:753-766):
   *   out = sqrt(a) * cond + sqrt(1 - a) * z,   a = aux1[l], l = (int)aux0[b]
   * aux0 = the per-clip labels (fp32 [B], the network's timestep input); aux1 = fp32 tables [3][i4] = alphas | k_cum |
   * theta_t of the i4-step schedule (a label outside [0, i4) gives NaN).  z is read from aux2 (NCHW, shaped like the
   * noised source) unless MCVD_F_PHILOX is set: then it is drawn in-kernel from Philox4x32-10 keyed by (seed, global
   * clip id, call ordinal, element) with w = int32 [4] = (seed lo, seed hi, first clip id, call ordinal) in device
   * memory, so one captured graph serves every call.  MCVD_F_GAMMA (with MCVD_F_PHILOX): z is the normalised Gamma
   * draw (g - k theta) / sqrt(1 - a), g ~ Gamma(k = k_cum[l], scale theta_t[l]) (k < 1 gives NaN). */
  MCVD_OP_NCHW_TO_NHWC = 1,
  /* [B,H,W,C0] NHWC -> [B,C0,H,W] NCHW (network output back to the reference layout).  C1 > 0: source
   * channel pitch (the last conv writes Cout padded to 16). */
  MCVD_OP_NHWC_TO_NCHW = 2,
  /* sinusoidal timestep embedding, layers.py:504-518.  src0 = t fp32 [B]; dst [B, Cout]. */
  MCVD_OP_TIMESTEP_EMBED = 3,
  /* dst[b,j] = bias[j] + sum_k act(src0[b,k]) * w[j,k]; w is nn.Linear layout [Cout, C0].
   * MCVD_F_ACT_IN applies SiLU to the input (temb MLP ncsnpp_more.py:278-280; every FiLM
   * projection Dense_0(act(temb)) layerspp.py:521).  B rows. */
  MCVD_OP_LINEAR = 4,
  /* GroupNorm statistics, pass 1: per (b, pixel-chunk, channel) sum / sum-of-squares in fp64.
   * src0 [B,H,W,C0] (+ src1 [B,H,W,C1], virtual channel concat); dst = double2 [B, i0, C0+C1],
   * i0 = number of pixel chunks. */
  MCVD_OP_GN_PARTIAL = 5,
  /* GroupNorm statistics, pass 2 + FiLM/affine folding: reduces the partials over chunks and over
   * the i1 = C/groups channels of a group (groups are contiguous channel ranges,
   * layerspp.py:474-477), and writes one float4 per (b, channel): (mean, rstd, G, S) so that the
   * consumer computes  y = ((x - mean) * rstd [*(1+gamma)+beta]) * G + S.
   *   aux0 != NULL, MCVD_F_FILM : G = 1 + aux0[b*i2 + i3 + c], S = aux0[b*i2 + i3 + C + c]
   *                               (scale/shift = chunk(Dense_0(act(temb)), 2), layerspp.py:521-523,536)
   *   aux0 != NULL, !FILM       : G = aux0[c] (GroupNorm weight), S = aux1[c] (bias)
   *   aux0 == NULL              : G = 1, S = 0
   * src0 = per-channel partials of the first tensor ([B,i0,C0]); src1/C1 = partials of a second tensor
   * (virtual concat) or NULL/0; i0 = chunks, f0 = eps.  Partials are per TENSOR, so a tensor consumed by
   * several norms (skip connections) is scanned once.
   * i4 / i5 != 0: src0 / src1 is not a chunk array but the int64 tile statistics a MCVD_OP_CONV_UMMA2
   * epilogue wrote for that tensor, i4 / i5 = kernel size (1|3) of the producing conv (fixes the tile geometry).
   * dst2 != NULL additionally receives the planar table [B][3][C] = mean | rstd*G | S read by
   * MCVD_OP_CONV_UMMA2. */
  MCVD_OP_GN_FINALIZE = 6,
  /* normalise + FiLM (+ SPADE gamma/beta) + SiLU + optional 4x4 FIR up/down-sampling, fp32 NHWC in
   * and out.  get_act_norm.forward layerspp.py:518-549, MySPADE.forward :152-173 (norm part),
   * upsample_2d / downsample_2d up_or_down_sampling.py:196-258 == upfirdn2d.  H,W are OUTPUT
   * dims; src0/src1 are the (virtually concatenated) inputs at input resolution; aux0 = float4
   * table from GN_FINALIZE (NULL = raw pass-through, used for the skip branch FIR(x));
   * aux1/aux2 = SPADE gamma/beta [B,Hin,Win,C] or NULL.  dst2 != NULL additionally receives the same
   * resampling of the RAW input (the skip branch FIR(x) of up/down blocks, layerspp.py:600-611) so the
   * input is read once. */
  MCVD_OP_APPLY = 7,
  /* direct convolution as implicit GEMM on CUDA cores (fp32 FFMA), NHWC.  nn.Conv2d 3x3 pad 1 /
   * 1x1 (layers.py:89-113) and NIN (layers.py:541-544).  i0 = ksize (1|3); src0/src1 virtual
   * concat; w = packed [taps][C0+C1][i1] fp32 (i1 = Cout rounded up to 4); bias [Cout];
   * aux0 = residual [B,H,W,Cout] or NULL; dst = f0 * (conv + bias + residual);
   * MCVD_F_ACT_OUT applies SiLU to the result (SPADE mlp_shared, layerspp.py:148). */
  MCVD_OP_CONV_SIMT = 8,
  /* softmax(q.k^T * f0) v over all H*W keys, per (b, head); AttnBlockpp.forward layerspp.py:239-245.
   * src0 = qkv [B, T, 3*C0] (q | k | v along channels), i0 = heads, i1 = head dim, T = H*W;
   * dst [B, T, C0]. */
  MCVD_OP_ATTENTION = 9,
  /* nearest-neighbour resize of an NHWC map (F.interpolate(segmap, 'nearest'), layerspp.py:165).
   * src0 [B, i0, i1, C0] -> dst [B, H, W, C0]. */
  MCVD_OP_RESIZE_NEAREST = 10,
  /* reverse-diffusion update on the NCHW state, in place (models/__init__.py:287-290,324-333 for
   * DDPM; :163-166 DDIM; denoise :331-333):
   *   x0 = f0 * (x - f1 * eps);  if MCVD_F_CLIP: x0 = clamp(x0,-1,1);
   *   x  = f2 * x0 + f3 * x + f4 * eps + f5 * z
   * dst = x [B,C0,H,W] NCHW (in place); src0 = eps [B,H,W,C0] NHWC (channel pitch Cout if > 0); src1 = z NCHW or NULL
   * (MCVD_F_PHILOX: z from Philox4x32-10 keyed by (seed=i0|i1<<32, clip id = i2 + b, step = i3)).
   * MCVD_F_GAMMA: z is the centred Gamma draw g - k theta, g ~ Gamma(shape k = f6, scale theta = f7), drawn in-kernel
   * with the same key fields in its own Philox domain (models/__init__.py:319-322, Gamma diffusion noise).  The
   * caller folds any normalisation (the reference's 1 / sqrt(1 - alpha)) into f5.  Marsaglia-Tsang with the centred
   * value formed without cancellation (at k = 2.5e10 the mean k theta is 1.6e5 standard deviations away from 0) and
   * the acceptance test in fp64; after 16 rejections in a row (probability < 1e-20 for k >= 1) z = 0, the mean.
   * The launch rejects k < 1 and theta <= 0. */
  MCVD_OP_DIFFUSION_UPDATE = 11,
  /* 3x3 / 1x1 convolution on the 5th-gen tensor cores (tcgen05.mma kind::f16, fp16 hi/lo split of
   * both operands, fp32 accumulation in TMEM), with the GroupNorm/FiLM/SiLU transform of the input
   * fused into the shared-memory staging.  Same semantics as MCVD_OP_CONV_SIMT; see
   * mcvd_b200/csrc/conv_umma.cu.  aux1 = norm table of (src0|src1) or NULL; i1 = n tile; i2 = accumulators
   * per tile (0 = auto); i3 = operand split for accuracy experiments (0 | 3 = all three products, 1 = drop
   * hi*lo_w, 2 = drop lo_a*hi, 4 = hi*hi only); f1 = weight un-scale.  Optional second K-segment (src2|src3 with C2|C3 channels, RAW,
   * centre tap only, weights appended per n-tile): the 1x1 shortcut Conv_2(x) of ResnetBlockBigGANpp
   * (layerspp.py:618-619) accumulated into the same TMEM tile as Conv_1, so
   * dst = f0 * (Conv_1(act(norm(h))) + Conv_2(x) + bias + residual) in ONE kernel.
   * dst2 = NULL, or the int64 tile statistics of the stored output (format and meaning as in MCVD_OP_CONV_UMMA2:
   * [tiles][NJ][2][Cout], mcvd_umma2_stats_bytes() bytes) for the GroupNorm that reads dst next;
   * aux2 = NULL or int64 [grid][16] cycle counters (tools/umma_timing.py).
   * Kernel size 1 without a second segment and without dst2 (NIN / q,k,v / skip projections,
   * layers.py:541-556, layerspp.py:230-249,618-619) is served by the input-stationary kernel of
   * mcvd_b200/csrc/conv1x1_umma.cu (same weights, bit-identical results) when the channel counts are multiples
   * of 32 and, with a norm table, the maps hold >= 64 positions; MCVD_CONV1X1=0 in the environment disables it. */
  MCVD_OP_CONV_UMMA = 12,
  /* final 3x3 conv with tiny Cout (<= 16) and fused input norm: conv3x3(SiLU(GN(x))) of
   * ncsnpp_more.py:375-379; aux0 = float4 norm table or NULL. */
  MCVD_OP_CONV_SMALLN = 13,
  /* dst[i] = src0[i] (i0 floats) -- device-to-device copy inside a program. */
  MCVD_OP_COPY = 14,
  /* MCVD_OP_ATTENTION on the tensor cores (tcgen05, fp16 hi/lo split, flash-style online softmax with
   * S and the per-tile P.V product in TMEM); same fields plus dst2 = device scratch of at least
   * mcvd_attention_scratch_bytes(B, H*W, C0) bytes (16-byte aligned): a first kernel splits q, k, v into
   * fp16 hi/lo operand images there, the attention kernel streams them in with cp.async.bulk (2 launches).
   * Head dim in {32,48,64,96,128,192}, H*W a multiple of the key tile (128; 64 for head dim 128; 32 for head
   * dim 192; H*W itself when smaller).  See mcvd_b200/csrc/attention_umma.cu. */
  MCVD_OP_ATTENTION_UMMA = 15,
  /* MCVD_OP_CONV_UMMA on CTA pairs (tcgen05.mma.cta_group::2, M = 256 over the two SMs of a TPC; see
   * mcvd_b200/csrc/conv_umma2.cu).  Same semantics and fields, except:
   *   aux1 = norm table of (src0|src1) in the planar layout [B][3][C0+C1] = mean | rstd*G | S that
   *          MCVD_OP_GN_FINALIZE writes to its dst2 (NULL: raw input);
   *   w    = weights packed by mcvd_umma2_pack_weights for n tile i1 and K-block i2
   *          (i2 = mcvd_umma2_plan(...); 0 skips the consistency check);
   *   i3   = operand split: 3 (default, also 0) = hi*hi + lo*hi + hi*lo, 1 = drop hi*lo (fp16 weights),
   *          2 = drop lo*hi (fp16 activations), 4 = hi*hi only -- accuracy experiments, DESIGN.md section 4;
   *   dst2 = NULL, or int64 [tiles][NJ][2][Cout] receiving the GroupNorm partial sums of the stored output
   *          (sum and sum of squares of round(x * 2^16), exact integer arithmetic; tiles = 128-position row
   *          tiles of the padded-flat position space, NJ = 127 / Pimg + 2 image slots per tile,
   *          mcvd_umma2_stats_bytes() bytes) -- nn.GroupNorm statistics of the NEXT act-norm
   *          (layerspp.py:474-477) without re-reading the activation;
   *   aux2 = NULL or int64 [grid][16] cycle counters (tools/umma_timing.py). */
  MCVD_OP_CONV_UMMA2 = 16,
  /* per-frame quality metrics of generated clips on the GPU (reference runners/ncsn_runner.py:1581-1600, which
   * loops over PIL images on the CPU): src0 = pred, src1 = real, both [B, C0*i0, H, W] fp32 in [0,1] (i0 frames of
   * C0 = 1|3 channels); dst = float64 [B, i0, 2] = (MSE over the frame's C0*H*W values, SSIM).  SSIM as the
   * reference calls it: skimage structural_similarity(data_range=255, gaussian_weights=True,
   * use_sample_covariance=False) on the 8-bit grey images PIL makes (x*255 truncated; RGB -> L = (19595 R + 38470 G +
   * 7471 B + 32768) >> 16), i.e. 11x11 Gaussian (sigma 1.5) moments, mean over the interior cropped by 5 pixels.
   * MCVD_F_ROUND: round the [0,1] values first (the reference does for (Stochastic)MovingMNIST, :1596-1599). */
  MCVD_OP_FRAME_METRICS = 17,
  MCVD_OP__COUNT
};

/* ---- flags ---------------------------------------------------------------------------------- */
#define MCVD_F_ACT_IN   (1 << 0)   /* SiLU on the input (LINEAR)                                   */
#define MCVD_F_ACT_OUT  (1 << 1)   /* SiLU on the output (APPLY: after the norm; CONV: on result)  */
#define MCVD_F_UP       (1 << 2)   /* APPLY: FIR upsample x2   (input is H/2 x W/2)               */
#define MCVD_F_DOWN     (1 << 3)   /* APPLY: FIR downsample x2 (input is 2H x 2W)                 */
#define MCVD_F_FILM     (1 << 4)   /* GN_FINALIZE: aux0 is the FiLM table                          */
#define MCVD_F_CLIP     (1 << 5)   /* DIFFUSION_UPDATE: clamp x0 to [-1, 1]                        */
#define MCVD_F_PHILOX   (1 << 6)   /* DIFFUSION_UPDATE: draw z in-kernel                           */
#define MCVD_F_ROUND    (1 << 7)   /* FRAME_METRICS: round the images before the grey conversion   */
#define MCVD_F_GAMMA    (1 << 8)   /* DIFFUSION_UPDATE / NCHW_TO_NHWC: Gamma noise instead of normal */
#define MCVD_F_NOISE    (1 << 9)   /* NCHW_TO_NHWC: diffuse the conditioning frames (noise_in_cond)  */

typedef struct McvdOp {
  int32_t kind;
  int32_t flags;
  int32_t B, H, W;          /* batch and OUTPUT spatial size                                   */
  int32_t C0, C1;           /* channels of src0 / src1 (C1 = 0: no second source)               */
  int32_t Cout;
  int32_t i0, i1, i2, i3;   /* per-kind integers, see the kind's comment                         */
  float f0, f1, f2, f3, f4, f5, f6, f7;
  const void* src0;
  const void* src1;
  const void* w;
  const void* bias;
  const void* aux0;
  const void* aux1;
  const void* aux2;
  void* dst;
  void* dst2;
  /* second K-segment of MCVD_OP_CONV_UMMA (fused 1x1 shortcut, see the kind's comment); NULL/0 otherwise */
  const void* src2;
  const void* src3;
  int32_t C2, C3;
  int32_t i4, i5, i6, i7;   /* more per-kind integers (ABI v4)                                  */
} McvdOp;

/* Library / ABI identification. */
int mcvd_abi_version(void);
/* sizeof(McvdOp) as compiled -- the Python ctypes mirror asserts equality at load time. */
int mcvd_sizeof_op(void);
/* Text of the last error on the calling thread ("" if none). */
const char* mcvd_last_error(void);
/* Compute capability of the current device as major*10+minor (e.g. 100), or <0. */
int mcvd_device_arch(void);

/* Launch ops[0..n) in order on `stream` (a cudaStream_t).  No synchronisation, re-entrant, uses the
 * device of the calling thread's current CUDA context (torch.cuda.device).  Capturable in a CUDA
 * graph. */
int mcvd_run_program(const McvdOp* ops, int n, void* stream);

/* Validate a program on the host without launching (shapes, alignment, NULLs).  Works without a
 * GPU. */
int mcvd_validate_program(const McvdOp* ops, int n);

/* Number of kernel launches mcvd_run_program would issue for this program (bench.py's
 * gpu_launches). */
int mcvd_count_launches(const McvdOp* ops, int n);

/* Weight packing for MCVD_OP_CONV_UMMA (device -> device, on `stream`):
 * w_taps = fp32 [taps][Cin][Cout] (the CONV_SIMT layout without Cout padding); out = the fp16 hi/lo
 * shared-memory images consumed by the tensor-core kernel; returns bytes required when out == NULL.
 * scale_log2 receives the power-of-two pre-scale applied to the weights (undone in the epilogue). */
long long mcvd_umma_pack_weights(const float* w_taps, int taps, int Cin, int Cout, int n_tile, int k_block,
                                 void* out, int scale_log2, void* stream);
/* Channels per K-block (32, 16, or 0 = unsupported) the tensor-core conv uses for sources with C0 / C1
 * channels; the packed weights must be produced with the same value. */
int mcvd_umma_kblock(int C0, int C1);
/* MCVD_OP_CONV_UMMA2 planning: channels per K-block (32 | 16, 0 = unsupported) for a conv of kernel size ks on
 * H x W maps with sources of C0|C1 (+ shortcut C2|C3) channels, n tile `n_tile`, with / without epilogue
 * statistics (the shared-memory plan depends on all of them); the weights must be packed with this value. */
int mcvd_umma2_plan(int H, int W, int ks, int C0, int C1, int C2, int C3, int n_tile, int stats);
/* The shared-memory plan behind mcvd_umma2_plan (diagnostics / tests; host arithmetic only): out[0..7] = K-block,
 * slab rows, image stages, raw-ring stages, weight stages, image slots per tile, TMEM columns, dynamic shared
 * memory bytes.  Returns 0, or -1 when the conv cannot run on this kernel. */
int mcvd_umma2_plan_info(int H, int W, int ks, int C0, int C1, int C2, int C3, int n_tile, int stats, int* out);
/* Bytes of the dst2 statistics array of a MCVD_OP_CONV_UMMA2 op. */
long long mcvd_umma2_stats_bytes(int B, int H, int W, int ks, int Cout);
/* Weight packing for MCVD_OP_CONV_UMMA2.  w_taps = fp32 [taps][Cin][Cout]; every (n tile, K-block, tap) becomes
 * two shared-memory images (one per CTA of the pair, NT/2 output columns each).  A conv with a fused 1x1
 * shortcut is packed with two calls into the same `out`: the main conv with stage_off = 0 and the shortcut
 * with stage_off = (Cin_main / KB) * taps, both with per_unit = total stages of one n tile.  Returns the bytes
 * this call fills (taps*Cin*Cout*4); out == NULL only queries. */
long long mcvd_umma2_pack_weights(const float* w_taps, int taps, int Cin, int Cout, int n_tile, int k_block,
                                  void* out, int scale_log2, int stage_off, int per_unit, void* stream);
/* Bytes of dst2 scratch one MCVD_OP_ATTENTION_UMMA op with batch B, T = H*W tokens and C channels needs. */
long long mcvd_attention_scratch_bytes(int B, int T, int C);

#ifdef __cplusplus
}
#endif
#endif /* MCVD_B200_H */
