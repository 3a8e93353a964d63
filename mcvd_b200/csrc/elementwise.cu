// Memory-bound kernels of the MCVD sampling path: layout changes, timestep embedding, FiLM linears,
// GroupNorm statistics, the fused normalise/FiLM/SPADE/SiLU/FIR "apply" pass, nearest resize and
// the reverse-diffusion update.  All tensors fp32; activations NHWC.
#include "mcvd_common.cuh"

namespace mcvd {

// ------------------------------------------------------------------------------------------------
// counter-based noise: Philox4x32-10 (Salmon et al., SC'11) keyed by (seed, global clip id, step or call, element), so
// a clip draws the same noise whichever GPU owns it (multi-GPU equivalence, SURVEY.md section 8e)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t out[4]) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0;
    uint32_t hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += W0; k1 += W1;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// Philox domains (4th counter word): one per noise stream, so no two streams share a counter
constexpr uint32_t DOM_STEP_NORMAL = 0x4d435644u;   // 'MCVD' (per-step normal noise; unchanged since ABI v1)
constexpr uint32_t DOM_STEP_GAMMA = 0x4d434700u;    // 'MCG' + attempt
constexpr uint32_t DOM_COND_NORMAL = 0x4d435643u;   // 'MCVC'
constexpr uint32_t DOM_COND_GAMMA = 0x4d434300u;    // 'MCC' + attempt

__device__ __forceinline__ float philox_normal(uint32_t seed_lo, uint32_t seed_hi, uint32_t clip, uint32_t step,
                                               uint32_t elem) {
  uint32_t r[4];
  philox4x32_10(elem, clip, step, DOM_STEP_NORMAL, seed_lo, seed_hi, r);
  // Box-Muller on two 32-bit uniforms in (0,1]
  float u1 = ((float)r[0] + 1.0f) * 2.3283064365386963e-10f;
  float u2 = ((float)r[1] + 0.5f) * 2.3283064365386963e-10f;
  u1 = fminf(fmaxf(u1, 1e-12f), 1.0f);
  float rad = sqrtf(-2.0f * logf(u1));
  return rad * cospif(2.0f * u2);
}

// Gamma(k, 1) by Marsaglia-Tsang (ACM TOMS 26(3), 2000), returned CENTRED: g - k, in fp64.  The diffusion schedule
// reaches k = 2.5e10, where g - k formed from g in fp32 would be quantised to whole ulps of g (an ulp of the mean is
// several percent of the standard deviation sqrt(k)).  With d = k - 1/3, c = 1/sqrt(9d), v = (1 + c x)^3:
//   d v - k = sqrt(d) x (1 + c x + (c x)^2 / 3) - 1/3       (no cancellation),
// and the acceptance test log u < x^2/2 + d - d v + d log v is evaluated as x^2/2 + d (log1p(t) - t), t = v - 1, in
// fp64.  Every attempt draws from its own Philox counter (domain + attempt), so the result is a pure function of the
// key.  After GAMMA_MAX_TRIES rejections in a row (acceptance is > 0.95 per attempt for k >= 1, so this has
// probability < 1e-20) the mean, 0, is returned.
constexpr int GAMMA_MAX_TRIES = 16;

__device__ double philox_gamma_centred(uint32_t seed_lo, uint32_t seed_hi, uint32_t clip, uint32_t ctr, uint32_t elem,
                                       uint32_t domain, double k) {
  const double d = k - 1.0 / 3.0, sd = sqrt(d), c = 1.0 / (3.0 * sd);
  for (int it = 0; it < GAMMA_MAX_TRIES; ++it) {
    uint32_t r[4];
    philox4x32_10(elem, clip, ctr, domain + (uint32_t)it, seed_lo, seed_hi, r);
    const float u1 = fminf(fmaxf(((float)r[0] + 1.0f) * 2.3283064365386963e-10f, 1e-12f), 1.0f);
    const float u2 = ((float)r[1] + 0.5f) * 2.3283064365386963e-10f;
    const double x = (double)(sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2));
    const double e = c * x;
    if (e <= -1.0) continue;                                   // v <= 0
    const double t = e * (3.0 + e * (3.0 + e));                // v - 1
    const double u = ((double)r[2] + 0.5) * 2.3283064365386963e-10;
    if (log(u) < 0.5 * x * x + d * (log1p(t) - t)) return sd * x * (1.0 + e + e * e * (1.0 / 3.0)) - 1.0 / 3.0;
  }
  return 0.0;
}

// ------------------------------------------------------------------------------------------------
// NCHW (+NCHW) -> NHWC  /  NHWC -> NCHW
// ------------------------------------------------------------------------------------------------
__global__ void k_nchw_to_nhwc(const float* __restrict__ s0, const float* __restrict__ s1, float* __restrict__ dst,
                               int B, int HW, int C0, int C1, int pitch) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)B * HW) return;
  int b = (int)(i / HW), p = (int)(i % HW);
  int C = C0 + C1;
  float* d = dst + i * pitch;
  for (int c = 0; c < C0; ++c) d[c] = s0[((long long)b * C0 + c) * HW + p];
  for (int c = 0; c < C1; ++c) d[C0 + c] = s1[((long long)b * C1 + c) * HW + p];
  for (int c = C; c < pitch; ++c) d[c] = 0.f;          // zero channel padding (tensor-core K alignment)
}

// MCVD_F_NOISE variant: the conditioning source (src1 if C1 > 0, else src0) becomes sqrt(a) cond + sqrt(1 - a) z with
// a = alphas[label of the clip].  The products and the sum are rounded separately, as the reference's fp32 tensor
// expression is, so injected noise reproduces the reference bit for bit.
struct CondNoiseArgs {
  const float* labels;   // [B]
  const float* tab;      // [3][T]: alphas | k_cum | theta_t
  const float* z;        // NCHW noise of the conditioning source, or NULL (Philox)
  const int* ctl;        // seed lo, seed hi, first clip id, call ordinal
  int T, gamma;
};

__device__ __forceinline__ float cond_noised(const CondNoiseArgs& a, int b, int cn, int Cn, int HW, int p, float v) {
  const float lf = a.labels[b];
  const int l = (int)lf;
  if (!(lf >= 0.f) || l >= a.T) return __int_as_float(0x7fffffff);        // label outside the schedule: NaN
  const float al = a.tab[l];
  float z;
  if (a.z) {
    z = a.z[((long long)b * Cn + cn) * HW + p];
  } else {
    const uint32_t clip = (uint32_t)(a.ctl[2] + b), call = (uint32_t)a.ctl[3], elem = (uint32_t)(cn * HW + p);
    if (a.gamma) {
      const double k = (double)a.tab[a.T + l], th = (double)a.tab[2 * a.T + l];
      if (!(k >= 1.0)) return __int_as_float(0x7fffffff);
      z = (float)(th * philox_gamma_centred((uint32_t)a.ctl[0], (uint32_t)a.ctl[1], clip, call, elem, DOM_COND_GAMMA, k) /
                  sqrt(1.0 - (double)al));
    } else {
      uint32_t r[4];
      philox4x32_10(elem, clip, call, DOM_COND_NORMAL, (uint32_t)a.ctl[0], (uint32_t)a.ctl[1], r);
      const float u1 = fminf(fmaxf(((float)r[0] + 1.0f) * 2.3283064365386963e-10f, 1e-12f), 1.0f);
      const float u2 = ((float)r[1] + 0.5f) * 2.3283064365386963e-10f;
      z = sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
    }
  }
  return __fadd_rn(__fmul_rn(sqrtf(al), v), __fmul_rn(sqrtf(1.0f - al), z));
}

__global__ void k_nchw_to_nhwc_noise(const float* __restrict__ s0, const float* __restrict__ s1, float* __restrict__ dst,
                                     int B, int HW, int C0, int C1, int pitch, CondNoiseArgs na) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)B * HW) return;
  int b = (int)(i / HW), p = (int)(i % HW);
  int C = C0 + C1;
  float* d = dst + i * pitch;
  for (int c = 0; c < C0; ++c) {
    const float v = s0[((long long)b * C0 + c) * HW + p];
    d[c] = C1 == 0 ? cond_noised(na, b, c, C0, HW, p, v) : v;
  }
  for (int c = 0; c < C1; ++c) d[C0 + c] = cond_noised(na, b, c, C1, HW, p, s1[((long long)b * C1 + c) * HW + p]);
  for (int c = C; c < pitch; ++c) d[c] = 0.f;
}

int launch_nchw_to_nhwc(const McvdOp& op, cudaStream_t s) {
  MCVD_CHECK(op.src0 && op.dst && (op.C1 == 0 || op.src1), "NCHW_TO_NHWC: null pointer");
  if (op.flags & MCVD_F_NOISE) {
    const bool philox = (op.flags & MCVD_F_PHILOX) != 0;
    MCVD_CHECK(op.aux0 && op.aux1 && op.i4 > 0, "NCHW_TO_NHWC noise: labels (aux0) and schedule tables (aux1, i4 entries) required");
    MCVD_CHECK(philox ? op.w != nullptr : op.aux2 != nullptr,
               "NCHW_TO_NHWC noise: %s", philox ? "MCVD_F_PHILOX needs the control block (w)" : "noise buffer (aux2) missing");
    MCVD_CHECK(!(op.flags & MCVD_F_GAMMA) || philox, "NCHW_TO_NHWC noise: MCVD_F_GAMMA draws in-kernel (needs MCVD_F_PHILOX)");
    CondNoiseArgs na{(const float*)op.aux0, (const float*)op.aux1, philox ? nullptr : (const float*)op.aux2,
                     (const int*)op.w, op.i4, (op.flags & MCVD_F_GAMMA) ? 1 : 0};
    long long n = (long long)op.B * op.H * op.W;
    k_nchw_to_nhwc_noise<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(
        (const float*)op.src0, (const float*)op.src1, (float*)op.dst, op.B, op.H * op.W, op.C0, op.C1,
        op.Cout > 0 ? op.Cout : op.C0 + op.C1, na);
    MCVD_CUDA_LAUNCH_CHECK("nchw_to_nhwc_noise");
    return 0;
  }
  long long n = (long long)op.B * op.H * op.W;
  k_nchw_to_nhwc<<<(unsigned)((n + 255) / 256), 256, 0, s>>>((const float*)op.src0, (const float*)op.src1,
                                                             (float*)op.dst, op.B, op.H * op.W, op.C0, op.C1,
                                                             op.Cout > 0 ? op.Cout : op.C0 + op.C1);
  MCVD_CUDA_LAUNCH_CHECK("nchw_to_nhwc");
  return 0;
}

__global__ void k_nhwc_to_nchw(const float* __restrict__ src, float* __restrict__ dst, int B, int HW, int C,
                               int pitch) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)B * HW) return;
  int b = (int)(i / HW), p = (int)(i % HW);
  const float* sp = src + i * pitch;
  for (int c = 0; c < C; ++c) dst[((long long)b * C + c) * HW + p] = sp[c];
}

int launch_nhwc_to_nchw(const McvdOp& op, cudaStream_t s) {
  MCVD_CHECK(op.src0 && op.dst, "NHWC_TO_NCHW: null pointer");
  long long n = (long long)op.B * op.H * op.W;
  k_nhwc_to_nchw<<<(unsigned)((n + 255) / 256), 256, 0, s>>>((const float*)op.src0, (float*)op.dst, op.B,
                                                             op.H * op.W, op.C0, op.C1 > 0 ? op.C1 : op.C0);
  MCVD_CUDA_LAUNCH_CHECK("nhwc_to_nchw");
  return 0;
}

__global__ void k_copy(const float* __restrict__ src, float* __restrict__ dst, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) dst[i] = src[i];
}

int launch_copy(const McvdOp& op, cudaStream_t s) {
  MCVD_CHECK(op.src0 && op.dst, "COPY: null pointer");
  long long n = (long long)op.i0 + ((long long)op.i1 << 31);
  unsigned g = (unsigned)((n + 255) / 256);
  if (g > 148 * 16) g = 148 * 16;
  if (g == 0) g = 1;
  k_copy<<<g, 256, 0, s>>>((const float*)op.src0, (float*)op.dst, n);
  MCVD_CUDA_LAUNCH_CHECK("copy");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// timestep embedding: dst[b, k] = sin(t_b * f_k), dst[b, half + k] = cos(t_b * f_k)
// f_k comes from the host (computed exactly as the reference does, layers.py:508-511) so the
// argument t*f is bit-identical to the reference's; only sinf/cosf differ (<= 2 ulp).
// ------------------------------------------------------------------------------------------------
__global__ void k_timestep_embed(const float* __restrict__ t, const float* __restrict__ freqs,
                                 float* __restrict__ dst, int B, int dim) {
  int half = dim / 2;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * dim) return;
  int b = i / dim, k = i % dim;
  float v = 0.f;
  if (k < half) v = sinf(t[b] * freqs[k]);
  else if (k < 2 * half) v = cosf(t[b] * freqs[k - half]);
  dst[i] = v;
}

int launch_timestep_embed(const McvdOp& op, cudaStream_t s) {
  MCVD_CHECK(op.src0 && op.w && op.dst, "TIMESTEP_EMBED: null pointer");
  int n = op.B * op.Cout;
  k_timestep_embed<<<cdiv(n, 256), 256, 0, s>>>((const float*)op.src0, (const float*)op.w, (float*)op.dst, op.B,
                                                op.Cout);
  MCVD_CUDA_LAUNCH_CHECK("timestep_embed");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// linear: dst[b, j] = act_out(bias[j] + sum_k act_in(src[b, k]) * w[j, k]);  one warp per output j
// ------------------------------------------------------------------------------------------------
constexpr int LIN_BT = 16;

__global__ void __launch_bounds__(128) k_linear(const float* __restrict__ src, const float* __restrict__ w,
                                                const float* __restrict__ bias, float* __restrict__ dst, int B,
                                                int K, int N, int flags) {
  int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int j = blockIdx.x * 4 + warp;
  if (j >= N) return;
  const float* wr = w + (long long)j * K;
  if (B == 1) {
    // uniform-timestep sampling: one row (the per-step FiLM projection is a 33k x 384 GEMV) -- stream the
    // weight row with 16-byte loads when it is aligned, one shuffle tree
    float acc = 0.f;
    if ((K & 3) == 0) {
      for (int k = lane * 4; k < K; k += 128) {
        const float4 wv = __ldg(reinterpret_cast<const float4*>(wr + k));
        float4 xv = *reinterpret_cast<const float4*>(src + k);
        if (flags & MCVD_F_ACT_IN) { xv.x = silu_f(xv.x); xv.y = silu_f(xv.y); xv.z = silu_f(xv.z); xv.w = silu_f(xv.w); }
        acc = fmaf(wv.x, xv.x, acc); acc = fmaf(wv.y, xv.y, acc); acc = fmaf(wv.z, xv.z, acc); acc = fmaf(wv.w, xv.w, acc);
      }
    } else {
      for (int k = lane; k < K; k += 32) {
        float xv = src[k];
        if (flags & MCVD_F_ACT_IN) xv = silu_f(xv);
        acc = fmaf(wr[k], xv, acc);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) {
      acc += bias ? bias[j] : 0.f;
      if (flags & MCVD_F_ACT_OUT) acc = silu_f(acc);
      dst[j] = acc;
    }
    return;
  }
  for (int b0 = 0; b0 < B; b0 += LIN_BT) {
    float acc[LIN_BT];
#pragma unroll
    for (int i = 0; i < LIN_BT; ++i) acc[i] = 0.f;
    for (int k = lane; k < K; k += 32) {
      float wv = wr[k];
#pragma unroll
      for (int i = 0; i < LIN_BT; ++i) {
        if (b0 + i < B) {
          float xv = src[(long long)(b0 + i) * K + k];
          if (flags & MCVD_F_ACT_IN) xv = silu_f(xv);
          acc[i] = fmaf(wv, xv, acc[i]);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < LIN_BT; ++i) {
      if (b0 + i >= B) break;                              // uniform across the warp
      float v = acc[i];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) {
        v += bias ? bias[j] : 0.f;
        if (flags & MCVD_F_ACT_OUT) v = silu_f(v);
        dst[(long long)(b0 + i) * N + j] = v;
      }
    }
  }
}

// Batched rows (per-clip timesteps: module.forward(x, labels) as the reference's own samplers call it).  The old path
// above evaluated act_in(src[b, k]) once per OUTPUT (33k x 64 x 384 SiLUs for the FiLM projection: 0.86 ms); here a
// block stages act_in of 16 batch rows in shared memory once and its 8 warps walk 64 output columns against them.
// Per-row arithmetic (k = lane*4 + 128*it, x,y,z,w in order, xor-shuffle tree) is exactly the single-row path's, so a
// batch of equal timesteps reproduces the uniform-timestep evaluation bit for bit.
constexpr int LIN_COLS = 64;

__global__ void __launch_bounds__(256) k_linear_batched(const float* __restrict__ src, const float* __restrict__ w,
                                                        const float* __restrict__ bias, float* __restrict__ dst, int B,
                                                        int K, int N, int flags) {
  extern __shared__ __align__(16) float lin_xs[];            // [LIN_BT][K]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int j0 = blockIdx.x * LIN_COLS;
  for (int b0 = 0; b0 < B; b0 += LIN_BT) {
    __syncthreads();                                         // previous tile's readers are done
    for (int i = threadIdx.x; i < LIN_BT * K; i += blockDim.x) {
      const int r = i / K, k = i - r * K;
      float xv = 0.f;
      if (b0 + r < B) {
        xv = src[(long long)(b0 + r) * K + k];
        if (flags & MCVD_F_ACT_IN) xv = silu_f(xv);
      }
      lin_xs[i] = xv;
    }
    __syncthreads();
    for (int c = warp; c < LIN_COLS; c += 8) {
      const int j = j0 + c;
      if (j >= N) break;
      const float* wr = w + (long long)j * K;
      float acc[LIN_BT];
#pragma unroll
      for (int i = 0; i < LIN_BT; ++i) acc[i] = 0.f;
      for (int k = lane * 4; k < K; k += 128) {
        const float4 wv = __ldg(reinterpret_cast<const float4*>(wr + k));
#pragma unroll
        for (int i = 0; i < LIN_BT; ++i) {
          const float4 xv = *reinterpret_cast<const float4*>(lin_xs + i * K + k);
          acc[i] = fmaf(wv.x, xv.x, acc[i]); acc[i] = fmaf(wv.y, xv.y, acc[i]);
          acc[i] = fmaf(wv.z, xv.z, acc[i]); acc[i] = fmaf(wv.w, xv.w, acc[i]);
        }
      }
      const float bj = bias ? bias[j] : 0.f;
#pragma unroll
      for (int i = 0; i < LIN_BT; ++i) {
        float v = acc[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0 && b0 + i < B) {
          v += bj;
          if (flags & MCVD_F_ACT_OUT) v = silu_f(v);
          dst[(long long)(b0 + i) * N + j] = v;
        }
      }
    }
  }
}

int launch_linear(const McvdOp& op, cudaStream_t s) {
  MCVD_CHECK(op.src0 && op.w && op.dst, "LINEAR: null pointer");
  const size_t xs_bytes = (size_t)LIN_BT * op.C0 * sizeof(float);
  if (op.B > 1 && (op.C0 & 3) == 0 && xs_bytes <= 48 * 1024 && (((uintptr_t)op.w | (uintptr_t)op.src0) & 15) == 0) {
    k_linear_batched<<<cdiv(op.Cout, LIN_COLS), 256, xs_bytes, s>>>((const float*)op.src0, (const float*)op.w,
                                                                     (const float*)op.bias, (float*)op.dst, op.B, op.C0,
                                                                     op.Cout, op.flags);
    MCVD_CUDA_LAUNCH_CHECK("linear");
    return 0;
  }
  k_linear<<<cdiv(op.Cout, 4), 128, 0, s>>>((const float*)op.src0, (const float*)op.w, (const float*)op.bias,
                                            (float*)op.dst, op.B, op.C0, op.Cout, op.flags);
  MCVD_CUDA_LAUNCH_CHECK("linear");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// GroupNorm statistics.  Pass 1: grid (chunks, B), 4 warps; a warp owns 32-channel blocks
// round-robin and walks the chunk's pixels (128 B coalesced per pixel).  Deterministic.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_gn_partial(const float* __restrict__ s0, const float* __restrict__ s1,
                                                    double2* __restrict__ part, int HW, int C0, int C1,
                                                    int nchunk, int ppc) {
  int b = blockIdx.y, chunk = blockIdx.x;
  int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int C = C0 + C1;
  int p0 = chunk * ppc, p1 = min(p0 + ppc, HW);
  for (int cb = warp * 32; cb < C; cb += 128) {
    int c = cb + lane;
    if (c >= C) continue;
    const float* src;
    int cs, cc;
    if (c < C0) { src = s0; cs = C0; cc = c; } else { src = s1; cs = C1; cc = c - C0; }
    const float* ptr = src + ((long long)b * HW + p0) * cs + cc;
    double ds = 0.0, dq = 0.0;
    int p = p0;
    // 8 independent loads in flight per lane; fp32 partials over 8 pixels, fp64 across groups
    for (; p + 8 <= p1; p += 8) {
      float v[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = __ldg(ptr + (long long)i * cs);
      ptr += 8LL * cs;
      float fs = 0.f, fq = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) { fs += v[i]; fq = fmaf(v[i], v[i], fq); }
      ds += (double)fs;
      dq += (double)fq;
    }
    for (; p < p1; ++p) {
      const float v = __ldg(ptr);
      ptr += cs;
      ds += (double)v;
      dq += (double)v * (double)v;
    }
    part[((long long)b * nchunk + chunk) * C + c] = make_double2(ds, dq);
  }
}

int launch_gn_partial(const McvdOp& op, cudaStream_t s) {
  MCVD_CHECK(op.src0 && op.dst && (op.C1 == 0 || op.src1), "GN_PARTIAL: null pointer");
  int HW = op.H * op.W;
  int nchunk = op.i0;
  MCVD_CHECK(nchunk >= 1, "GN_PARTIAL: chunks < 1");
  int ppc = cdiv(HW, nchunk);
  dim3 grid(nchunk, op.B);
  k_gn_partial<<<grid, 128, 0, s>>>((const float*)op.src0, (const float*)op.src1, (double2*)op.dst, HW, op.C0,
                                    op.C1, nchunk, ppc);
  MCVD_CUDA_LAUNCH_CHECK("gn_partial");
  return 0;
}

// Pass 2: grid (groups, B); reduce partials, emit (mean, rstd, G, S) per channel.
// A source is either a chunk array of k_gn_partial (double2 [B][nchunk][C]) or the int64 tile statistics a
// k_conv_umma2 epilogue wrote for that tensor ([tiles][NJ][2][C]: sum and sum of squares of round(x * 2^16) over
// the rows of one 128-position tile that belong to one image).  Integer sums are exact, so the statistics do not
// depend on where the image sits in the batch (clip sharding stays bit-exact).
struct GnSrc {
  const void* p;
  int C;          // channels of this tensor
  int ks;         // 0: chunk partials; 1 | 3: tile statistics of a conv with this kernel size
};

__device__ __forceinline__ void gn_tile_geometry(int ks, int H, int W, int& pimg, int& nj) {
  pimg = ks == 3 ? (H + 1) * (W + 1) : H * W;
  nj = 127 / pimg + 2;
}

__global__ void __launch_bounds__(128) k_gn_finalize(GnSrc s0, GnSrc s1, float4* __restrict__ tab,
                                                     float* __restrict__ tab3, const float* __restrict__ aux0,
                                                     const float* __restrict__ aux1, int B, int H, int W, int cg,
                                                     int nchunk, float eps, int film, int film_stride, int film_off) {
  const int g = blockIdx.x, b = blockIdx.y;
  const int C0 = s0.C, C = s0.C + s1.C, HW = H * W;
  double ds = 0.0, dq = 0.0;                         // chunk-partial contributions
  long long s1lo = 0, s1hi = 0;                      // tile statistics: 64-bit partials summed as 32-bit halves
  unsigned long long s2lo = 0, s2hi = 0;
  bool any_tiles = false;
  // the group's channels may straddle the two tensors of a virtual concat: per tensor, the (item, channel) pairs
  // are spread over all 128 threads (items = pixel chunks or 128-position tiles)
  for (int k = 0; k < 2; ++k) {
    const GnSrc& sr = k ? s1 : s0;
    const int base = k ? C0 : 0;                                   // first global channel of this tensor
    const int c_lo = max(g * cg, base) - base, c_hi = min(g * cg + cg, base + sr.C) - base;
    const int nc = c_hi - c_lo;
    if (nc <= 0) continue;
    if (sr.ks == 0) {
      const double2* part = reinterpret_cast<const double2*>(sr.p);
      for (int i = threadIdx.x; i < nchunk * nc; i += blockDim.x) {
        const int chunk = i / nc, cl = c_lo + i % nc;
        const double2 v = part[((long long)b * nchunk + chunk) * sr.C + cl];
        ds += v.x;
        dq += v.y;
      }
    } else {
      any_tiles = true;
      int pimg, nj;
      gn_tile_geometry(sr.ks, H, W, pimg, nj);
      const long long q0 = (long long)b * pimg, q1 = q0 + pimg - 1;
      const int t_lo = (int)(q0 >> 7), nt = (int)(q1 >> 7) - t_lo + 1;
      const long long* st = reinterpret_cast<const long long*>(sr.p);
      for (int i = threadIdx.x; i < nt * nc; i += blockDim.x) {
        const int t = t_lo + i / nc, cl = c_lo + i % nc;
        long long tb0 = ((long long)t << 7) / pimg;
        if (tb0 > B - 1) tb0 = B - 1;
        const int jj = b - (int)tb0;
        const long long* e = st + (((long long)t * nj + jj) * 2) * sr.C + cl;
        const long long v1 = e[0];
        const unsigned long long v2 = (unsigned long long)e[sr.C];
        s1lo += (long long)(v1 & 0xffffffffLL);
        s1hi += v1 >> 32;
        s2lo += v2 & 0xffffffffULL;
        s2hi += v2 >> 32;
      }
    }
  }
  __shared__ double shd[2][4];
  __shared__ long long shi[4][4];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ds += __shfl_xor_sync(0xffffffffu, ds, o);
    dq += __shfl_xor_sync(0xffffffffu, dq, o);
    s1lo += __shfl_xor_sync(0xffffffffu, s1lo, o);
    s1hi += __shfl_xor_sync(0xffffffffu, s1hi, o);
    s2lo += __shfl_xor_sync(0xffffffffu, s2lo, o);
    s2hi += __shfl_xor_sync(0xffffffffu, s2hi, o);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    shd[0][warp] = ds; shd[1][warp] = dq;
    shi[0][warp] = s1lo; shi[1][warp] = s1hi; shi[2][warp] = (long long)s2lo; shi[3][warp] = (long long)s2hi;
  }
  __syncthreads();
  ds = shd[0][0] + shd[0][1] + shd[0][2] + shd[0][3];
  dq = shd[1][0] + shd[1][1] + shd[1][2] + shd[1][3];
  if (any_tiles) {
    const long long a1lo = shi[0][0] + shi[0][1] + shi[0][2] + shi[0][3];
    const long long a1hi = shi[1][0] + shi[1][1] + shi[1][2] + shi[1][3];
    const unsigned long long a2lo = (unsigned long long)(shi[2][0] + shi[2][1] + shi[2][2] + shi[2][3]);
    const unsigned long long a2hi = (unsigned long long)(shi[3][0] + shi[3][1] + shi[3][2] + shi[3][3]);
    // hi * 2^32 and lo are exact doubles; their sum is one correctly rounded addition of the exact total
    ds += ((double)a1hi * 4294967296.0 + (double)a1lo) * (1.0 / 65536.0);
    dq += ((double)a2hi * 4294967296.0 + (double)a2lo) * (1.0 / 4294967296.0);
  }
  const double cnt = (double)HW * (double)cg;
  const double mean = ds / cnt;
  double var = dq / cnt - mean * mean;
  if (var < 0.0) var = 0.0;
  const float rstd = (float)(1.0 / sqrt(var + (double)eps));
  const float fmean = (float)mean;
  for (int ci = threadIdx.x; ci < cg; ci += blockDim.x) {
    const int c = g * cg + ci;
    float G = 1.f, S = 0.f;
    if (aux0) {
      if (film) {
        G = 1.f + aux0[(long long)b * film_stride + film_off + c];
        S = aux0[(long long)b * film_stride + film_off + C + c];
      } else {
        G = aux0[c];
        S = aux1[c];
      }
    }
    tab[(long long)b * C + c] = make_float4(fmean, rstd, G, S);
    if (tab3) {
      float* t3 = tab3 + (long long)b * 3 * C + c;
      t3[0] = fmean;
      t3[C] = rstd * G;
      t3[2 * C] = S;
    }
  }
}

int launch_gn_finalize(const McvdOp& op, cudaStream_t s) {
  MCVD_CHECK(op.src0 && op.dst, "GN_FINALIZE: null pointer");
  int C = op.C0 + op.C1, cg = op.i1;
  MCVD_CHECK(cg > 0 && C % cg == 0, "GN_FINALIZE: channels %d not divisible by group size %d", C, cg);
  MCVD_CHECK(op.C1 == 0 || op.src1, "GN_FINALIZE: second partial array missing");
  int film = (op.flags & MCVD_F_FILM) ? 1 : 0;
  MCVD_CHECK(!op.aux0 || film || op.aux1, "GN_FINALIZE: affine needs weight and bias");
  MCVD_CHECK((op.i4 == 0 || op.i4 == 1 || op.i4 == 3) && (op.i5 == 0 || op.i5 == 1 || op.i5 == 3),
             "GN_FINALIZE: source kinds (%d, %d) must be 0 (chunks), 1 or 3 (conv tile statistics)", op.i4, op.i5);
  for (int k = 0; k < 2; ++k) {
    const int ks = k ? op.i5 : op.i4;
    if (ks == 0 || (k && op.C1 == 0)) continue;
    const long long pimg = ks == 3 ? (long long)(op.H + 1) * (op.W + 1) : (long long)op.H * op.W;
    MCVD_CHECK(pimg >= 64, "GN_FINALIZE: tile statistics need images of >= 64 positions (%dx%d)", op.H, op.W);
  }
  MCVD_CHECK((op.i4 != 0 && (op.C1 == 0 || op.i5 != 0)) || op.i0 >= 1, "GN_FINALIZE: chunks < 1");
  GnSrc s0{op.src0, op.C0, op.i4}, s1{op.src1, op.C1, op.C1 > 0 ? op.i5 : 0};
  dim3 grid(C / cg, op.B);
  k_gn_finalize<<<grid, 128, 0, s>>>(s0, s1, (float4*)op.dst, (float*)op.dst2, (const float*)op.aux0,
                                     (const float*)op.aux1, op.B, op.H, op.W, cg, op.i0, op.f0, film, op.i2, op.i3);
  MCVD_CUDA_LAUNCH_CHECK("gn_finalize");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// apply: y = act( ((x - mean) * rstd [*(1+gamma)+beta]) * G + S ), optionally through the 4x4 FIR
// up/down-sampler (pointwise kernel: one thread = 4 consecutive channels of one pixel; resampling kernel below).
// FIR taps: outer([1,3,3,1])/64 (down) or /16 (up, gain 4) -- up_or_down_sampling.py:182-258.
// ------------------------------------------------------------------------------------------------
struct ApplyArgs {
  const float* s0;
  const float* s1;
  const float4* tab;
  const float* gam;
  const float* bet;
  float* dst;
  float* dst2;      // optional: the same resampling applied to the RAW input (skip branch of up/down blocks)
  int B, H, W, Hin, Win, C0, C1, flags;
};

__device__ __forceinline__ float4 apply_fetch(const ApplyArgs& a, int b, int yi, int xi, int c, const float4 t[4],
                                              float4& raw) {
  // value of the transformed input at input pixel (yi, xi), channels c..c+3 (zero outside); raw = untransformed
  raw = make_float4(0.f, 0.f, 0.f, 0.f);
  if (yi < 0 || yi >= a.Hin || xi < 0 || xi >= a.Win) return raw;
  long long pix = ((long long)b * a.Hin + yi) * a.Win + xi;
  float4 v;
  if (c < a.C0) v = *reinterpret_cast<const float4*>(a.s0 + pix * a.C0 + c);
  else v = *reinterpret_cast<const float4*>(a.s1 + pix * a.C1 + (c - a.C0));
  raw = v;
  if (a.tab) {
    float r[4] = {v.x, v.y, v.z, v.w};
    float gm[4] = {0.f, 0.f, 0.f, 0.f}, bt[4] = {0.f, 0.f, 0.f, 0.f};
    if (a.gam) {
      int C = a.C0 + a.C1;
      float4 g4 = *reinterpret_cast<const float4*>(a.gam + pix * C + c);
      float4 b4 = *reinterpret_cast<const float4*>(a.bet + pix * C + c);
      gm[0] = g4.x; gm[1] = g4.y; gm[2] = g4.z; gm[3] = g4.w;
      bt[0] = b4.x; bt[1] = b4.y; bt[2] = b4.z; bt[3] = b4.w;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float n = (r[i] - t[i].x) * t[i].y;
      if (a.gam) n = n * (1.f + gm[i]) + bt[i];
      n = n * t[i].z + t[i].w;
      if (a.flags & MCVD_F_ACT_OUT) n = silu_f(n);
      r[i] = n;
    }
    v = make_float4(r[0], r[1], r[2], r[3]);
  }
  return v;
}

__device__ __forceinline__ void fma4(float4& acc, float w, const float4& v) {
  acc.x = fmaf(w, v.x, acc.x);
  acc.y = fmaf(w, v.y, acc.y);
  acc.z = fmaf(w, v.z, acc.z);
  acc.w = fmaf(w, v.w, acc.w);
}

__global__ void __launch_bounds__(256) k_apply(ApplyArgs a) {
  // pointwise form (no resampling): one thread = 4 consecutive channels of one pixel
  int C = a.C0 + a.C1;
  int C4 = C >> 2;
  long long total = (long long)a.B * a.H * a.W * C4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % C4) * 4;
    long long pix = i / C4;
    int x = (int)(pix % a.W);
    int y = (int)((pix / a.W) % a.H);
    int b = (int)(pix / ((long long)a.W * a.H));
    float4 t[4];
    if (a.tab) {
#pragma unroll
      for (int k = 0; k < 4; ++k) t[k] = a.tab[(long long)b * C + c + k];
    }
    float4 rw;
    float4 out = apply_fetch(a, b, y, x, c, t, rw);
    if (a.dst2) *reinterpret_cast<float4*>(a.dst2 + pix * C + c) = rw;
    *reinterpret_cast<float4*>(a.dst + pix * C + c) = out;
  }
}

// Resampling form.  A CTA owns (sample, output tile, 32-channel chunk): it transforms the input tile
// (+ FIR halo) ONCE into shared memory -- transformed and raw copies -- and every output pixel then
// takes its 4 (up) or 16 (down) taps from there.  The pointwise form above re-did the transform
// (two MUFU per element) for every tap; this one reads each input element once from HBM and keeps
// global accesses in 128-byte rows (8 lanes x float4 per pixel).
//   up:   16x16 outputs <- 10x10 inputs (8x8 + 1 halo);  even y=2a: (in[a-1] + 3 in[a])/4, odd: (3 in[a] + in[a+1])/4
//   down: 4x8 outputs   <- 10x18 inputs;                 out[y,x] = sum_ij k_i k_j / 64 * in[2y+i-1, 2x+j-1]
constexpr int RS_LANES = 8;                 // float4 lanes per pixel = 32 channels per CTA
template <bool UP>
struct RsTile {
  static constexpr int OH = UP ? 16 : 4, OW = UP ? 16 : 8;
  static constexpr int IH = UP ? 10 : 10, IW = UP ? 10 : 18;
};

template <bool UP>
__global__ void __launch_bounds__(256) k_apply_resample(ApplyArgs a, int tiles_x) {
  using T = RsTile<UP>;
  extern __shared__ float4 rs_smem[];
  float4* sT = rs_smem;                                   // [IH*IW][8] transformed
  float4* sR = rs_smem + T::IH * T::IW * RS_LANES;        // [IH*IW][8] raw (only when dst2)
  const int C = a.C0 + a.C1;
  const int b = blockIdx.z;
  const int ty = blockIdx.x / tiles_x, tx = blockIdx.x % tiles_x;
  const int lane = threadIdx.x & (RS_LANES - 1);
  const int c = (blockIdx.y * RS_LANES + lane) * 4;
  const bool c_ok = c < C;
  const int iy0 = UP ? ty * (T::OH / 2) - 1 : ty * (T::OH * 2) - 1;
  const int ix0 = UP ? tx * (T::OW / 2) - 1 : tx * (T::OW * 2) - 1;
  float4 t[4];
  if (a.tab && c_ok) {
#pragma unroll
    for (int k = 0; k < 4; ++k) t[k] = a.tab[(long long)b * C + c + k];
  }
  const bool want_raw = a.dst2 != nullptr;
#pragma unroll 4
  for (int px = threadIdx.x >> 3; px < T::IH * T::IW; px += 256 / RS_LANES) {
    int ly = px / T::IW, lx = px - ly * T::IW;
    float4 rw = make_float4(0.f, 0.f, 0.f, 0.f), v = rw;
    if (c_ok) v = apply_fetch(a, b, iy0 + ly, ix0 + lx, c, t, rw);
    sT[px * RS_LANES + lane] = v;
    if (want_raw) sR[px * RS_LANES + lane] = rw;
  }
  __syncthreads();
  if (!c_ok) return;
  for (int op = threadIdx.x >> 3; op < T::OH * T::OW; op += 256 / RS_LANES) {
    int oy = op / T::OW, ox = op - oy * T::OW;
    int Y = ty * T::OH + oy, X = tx * T::OW + ox;
    if (Y >= a.H || X >= a.W) continue;
    float4 out = make_float4(0.f, 0.f, 0.f, 0.f), out2 = out;
    if (UP) {
      // local rows r0, r0+1 with weights (1,3) for even outputs and (3,1) for odd ones
      int r0 = (oy >> 1) + (oy & 1), q0 = (ox >> 1) + (ox & 1);
      float wy0 = (oy & 1) ? 3.f : 1.f, wx0 = (ox & 1) ? 3.f : 1.f;
      float wy[2] = {wy0, 4.f - wy0}, wx[2] = {wx0, 4.f - wx0};
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          int p = ((r0 + i) * T::IW + q0 + j) * RS_LANES + lane;
          float w = wy[i] * wx[j] * (1.f / 16.f);
          fma4(out, w, sT[p]);
          if (want_raw) fma4(out2, w, sR[p]);
        }
    } else {
      const float kw[4] = {1.f, 3.f, 3.f, 1.f};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          int p = ((2 * oy + i) * T::IW + 2 * ox + j) * RS_LANES + lane;
          float w = kw[i] * kw[j] * (1.f / 64.f);
          fma4(out, w, sT[p]);
          if (want_raw) fma4(out2, w, sR[p]);
        }
    }
    long long pix = ((long long)b * a.H + Y) * a.W + X;
    if (want_raw) *reinterpret_cast<float4*>(a.dst2 + pix * C + c) = out2;
    *reinterpret_cast<float4*>(a.dst + pix * C + c) = out;
  }
}

template <bool UP>
static void launch_resample(const ApplyArgs& a, cudaStream_t s) {
  using T = RsTile<UP>;
  int C = a.C0 + a.C1;
  int tiles_x = (a.W + T::OW - 1) / T::OW, tiles_y = (a.H + T::OH - 1) / T::OH;
  dim3 grid(tiles_x * tiles_y, (C / 4 + RS_LANES - 1) / RS_LANES, a.B);
  size_t smem = (size_t)T::IH * T::IW * RS_LANES * sizeof(float4) * 2;
  k_apply_resample<UP><<<grid, 256, smem, s>>>(a, tiles_x);
}

int launch_apply(const McvdOp& op, cudaStream_t s) {
  MCVD_CHECK(op.src0 && op.dst && (op.C1 == 0 || op.src1), "APPLY: null pointer");
  MCVD_CHECK(op.C0 % 4 == 0 && op.C1 % 4 == 0, "APPLY: channels must be multiples of 4 (%d, %d)", op.C0, op.C1);
  MCVD_CHECK(!(op.aux1) || (op.aux2 && op.aux0), "APPLY: SPADE needs gamma, beta and the norm table");
  MCVD_CHECK(!((op.flags & MCVD_F_DOWN) && (op.flags & MCVD_F_UP)), "APPLY: both UP and DOWN set");
  ApplyArgs a;
  a.s0 = (const float*)op.src0; a.s1 = (const float*)op.src1; a.tab = (const float4*)op.aux0;
  a.gam = (const float*)op.aux1; a.bet = (const float*)op.aux2; a.dst = (float*)op.dst; a.dst2 = (float*)op.dst2;
  a.B = op.B; a.H = op.H; a.W = op.W; a.C0 = op.C0; a.C1 = op.C1; a.flags = op.flags;
  a.Hin = op.H; a.Win = op.W;
  if (op.B <= 0 || op.H <= 0 || op.W <= 0 || op.C0 + op.C1 <= 0) return 0;
  if (op.flags & MCVD_F_DOWN) {
    MCVD_CHECK(op.B <= 65535, "APPLY: batch too large for the resampling grid (%d)", op.B);
    a.Hin = op.H * 2; a.Win = op.W * 2;
    launch_resample<false>(a, s);
  } else if (op.flags & MCVD_F_UP) {
    MCVD_CHECK(op.H % 2 == 0 && op.W % 2 == 0, "APPLY: upsample output must be even");
    MCVD_CHECK(op.B <= 65535, "APPLY: batch too large for the resampling grid (%d)", op.B);
    a.Hin = op.H / 2; a.Win = op.W / 2;
    launch_resample<true>(a, s);
  } else {
    long long total = (long long)op.B * op.H * op.W * ((op.C0 + op.C1) / 4);
    long long blocks = (total + 255) / 256;
    if (blocks > 148LL * 32) blocks = 148LL * 32;
    k_apply<<<(unsigned)blocks, 256, 0, s>>>(a);
  }
  MCVD_CUDA_LAUNCH_CHECK("apply");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// nearest resize (F.interpolate(mode='nearest'): src index = floor(dst index * in / out))
// ------------------------------------------------------------------------------------------------
__global__ void k_resize_nearest(const float* __restrict__ src, float* __restrict__ dst, int B, int Hin, int Win,
                                 int H, int W, int C) {
  long long total = (long long)B * H * W * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % C);
    long long pix = i / C;
    int x = (int)(pix % W), y = (int)((pix / W) % H), b = (int)(pix / ((long long)W * H));
    // PyTorch 'nearest': src = min(floor(dst * scale), in - 1), scale = in / out (float)
    float sy = (float)Hin / (float)H, sx = (float)Win / (float)W;
    int yi = min((int)floorf(y * sy), Hin - 1), xi = min((int)floorf(x * sx), Win - 1);
    dst[i] = src[(((long long)b * Hin + yi) * Win + xi) * C + c];
  }
}

int launch_resize_nearest(const McvdOp& op, cudaStream_t s) {
  MCVD_CHECK(op.src0 && op.dst, "RESIZE_NEAREST: null pointer");
  long long total = (long long)op.B * op.H * op.W * op.C0;
  long long blocks = (total + 255) / 256;
  if (blocks > 148LL * 32) blocks = 148LL * 32;
  k_resize_nearest<<<(unsigned)blocks, 256, 0, s>>>((const float*)op.src0, (float*)op.dst, op.B, op.i0, op.i1, op.H,
                                                    op.W, op.C0);
  MCVD_CUDA_LAUNCH_CHECK("resize_nearest");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// reverse-diffusion update (DDPM / DDIM / denoise), optional in-kernel Philox4x32-10 normal or centred Gamma noise.
// ------------------------------------------------------------------------------------------------
__global__ void k_diffusion_update(float* __restrict__ x, const float* __restrict__ eps, const float* __restrict__ z,
                                   int B, int C, int HW, int pitch, float k0, float k1, float ca, float cb, float cc,
                                   float sigma, int flags, uint32_t seed_lo, uint32_t seed_hi, int clip0, int step,
                                   double gk, double gtheta) {
  long long total = (long long)B * C * HW;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int p = (int)(i % HW);
  int c = (int)((i / HW) % C);
  int b = (int)(i / ((long long)HW * C));
  float xv = x[i];
  float ev = eps[((long long)b * HW + p) * pitch + c];
  float x0 = k0 * (xv - k1 * ev);
  if (flags & MCVD_F_CLIP) x0 = fminf(fmaxf(x0, -1.f), 1.f);
  float r = ca * x0 + cb * xv;
  if (cc != 0.f) r += cc * ev;
  if (sigma != 0.f) {
    float zv;
    if (flags & MCVD_F_GAMMA)
      zv = (float)(gtheta * philox_gamma_centred(seed_lo, seed_hi, (uint32_t)(clip0 + b), (uint32_t)step,
                                                 (uint32_t)(c * HW + p), DOM_STEP_GAMMA, gk));
    else if (flags & MCVD_F_PHILOX) zv = philox_normal(seed_lo, seed_hi, (uint32_t)(clip0 + b), (uint32_t)step, (uint32_t)(c * HW + p));
    else zv = z[i];
    r += sigma * zv;
  }
  x[i] = r;
}

int launch_diffusion_update(const McvdOp& op, cudaStream_t s) {
  MCVD_CHECK(op.src0 && op.dst, "DIFFUSION_UPDATE: null pointer");
  MCVD_CHECK(op.f5 == 0.f || (op.flags & (MCVD_F_PHILOX | MCVD_F_GAMMA)) || op.src1, "DIFFUSION_UPDATE: sigma != 0 needs noise");
  MCVD_CHECK(!(op.flags & MCVD_F_GAMMA) || (op.f6 >= 1.f && op.f7 > 0.f),
             "DIFFUSION_UPDATE: Gamma noise needs shape k >= 1 and scale theta > 0 (got k = %g, theta = %g)", op.f6, op.f7);
  long long total = (long long)op.B * op.C0 * op.H * op.W;
  k_diffusion_update<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(
      (float*)op.dst, (const float*)op.src0, (const float*)op.src1, op.B, op.C0, op.H * op.W,
      op.Cout > 0 ? op.Cout : op.C0, op.f0, op.f1, op.f2,
      op.f3, op.f4, op.f5, op.flags, (uint32_t)op.i0, (uint32_t)op.i1, op.i2, op.i3, (double)op.f6, (double)op.f7);
  MCVD_CUDA_LAUNCH_CHECK("diffusion_update");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// per-frame MSE and SSIM of generated clips (see MCVD_OP_FRAME_METRICS in include/mcvd_b200.h).
// grid (frames, B); one CTA holds the two 8-bit grey images in shared memory and evaluates the 11x11 Gaussian
// moments of every interior pixel in fp64 (the interior crop of 5 pixels is exactly the filter radius, so the
// 'reflect' boundary mode of scipy's gaussian_filter never enters the mean).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_frame_metrics(const float* __restrict__ pred, const float* __restrict__ real,
                                                       double* __restrict__ out, int C, int nf, int H, int W,
                                                       int round_first) {
  extern __shared__ float gm_smem[];
  float* gx = gm_smem;                 // pred, grey 0..255
  float* gy = gm_smem + H * W;         // real
  __shared__ double red[2][8];
  const int f = blockIdx.x, b = blockIdx.y, HW = H * W;
  const float* p0 = pred + ((long long)b * nf + f) * C * HW;
  const float* r0 = real + ((long long)b * nf + f) * C * HW;
  double se = 0.0;
  for (int i = threadIdx.x; i < HW; i += blockDim.x) {
    int pb[3], rb[3];
    for (int c = 0; c < C; ++c) {
      float pv = p0[c * HW + i], rv = r0[c * HW + i];
      const double d = (double)rv - (double)pv;
      se += d * d;
      if (round_first) { pv = rintf(pv); rv = rintf(rv); }          // torch.round: half to even
      pb[c] = (int)(unsigned char)(int)(pv * 255.0f);               // ToPILImage: mul(255).byte()
      rb[c] = (int)(unsigned char)(int)(rv * 255.0f);
    }
    if (C == 1) { gx[i] = (float)pb[0]; gy[i] = (float)rb[0]; }
    else {
      gx[i] = (float)((pb[0] * 19595 + pb[1] * 38470 + pb[2] * 7471 + 0x8000) >> 16);   // PIL RGB -> L
      gy[i] = (float)((rb[0] * 19595 + rb[1] * 38470 + rb[2] * 7471 + 0x8000) >> 16);
    }
  }
  __syncthreads();
  // 1-D Gaussian, sigma 1.5, radius 5, normalised (scipy.ndimage._gaussian_kernel1d)
  double g[11];
  {
    double sum = 0.0;
    for (int k = -5; k <= 5; ++k) { g[k + 5] = exp(-0.5 * (double)(k * k) / 2.25); sum += g[k + 5]; }
    for (int k = 0; k < 11; ++k) g[k] /= sum;
  }
  const double C1 = (0.01 * 255.0) * (0.01 * 255.0), C2 = (0.03 * 255.0) * (0.03 * 255.0);
  const int ih = H - 10, iw = W - 10;
  double ssum = 0.0;
  for (int i = threadIdx.x; i < ih * iw; i += blockDim.x) {
    const int y = i / iw + 5, x = i % iw + 5;
    double ux = 0, uy = 0, uxx = 0, uyy = 0, uxy = 0;
    for (int dy = -5; dy <= 5; ++dy) {
      double rx = 0, ry = 0, rxx = 0, ryy = 0, rxy = 0;
      const float* px = gx + (y + dy) * W + x, *py = gy + (y + dy) * W + x;
#pragma unroll
      for (int dx = -5; dx <= 5; ++dx) {
        const double a = px[dx], c = py[dx], w = g[dx + 5];
        rx += w * a; ry += w * c; rxx += w * a * a; ryy += w * c * c; rxy += w * a * c;
      }
      const double w = g[dy + 5];
      ux += w * rx; uy += w * ry; uxx += w * rxx; uyy += w * ryy; uxy += w * rxy;
    }
    const double vx = uxx - ux * ux, vy = uyy - uy * uy, vxy = uxy - ux * uy;
    ssum += ((2 * ux * uy + C1) * (2 * vxy + C2)) / ((ux * ux + uy * uy + C1) * (vx + vy + C2));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    se += __shfl_xor_sync(0xffffffffu, se, o);
    ssum += __shfl_xor_sync(0xffffffffu, ssum, o);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { red[0][warp] = se; red[1][warp] = ssum; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0, c = 0;
    for (int w = 0; w < 8; ++w) { a += red[0][w]; c += red[1][w]; }
    out[((long long)b * nf + f) * 2 + 0] = a / ((double)C * HW);
    out[((long long)b * nf + f) * 2 + 1] = (ih > 0 && iw > 0) ? c / ((double)ih * iw) : 0.0;
  }
}

int launch_frame_metrics(const McvdOp& op, cudaStream_t s) {
  MCVD_CHECK(op.src0 && op.src1 && op.dst, "FRAME_METRICS: null pointer");
  MCVD_CHECK(op.C0 == 1 || op.C0 == 3, "FRAME_METRICS: %d channels per frame (1 or 3)", op.C0);
  MCVD_CHECK(op.i0 >= 1 && op.H >= 11 && op.W >= 11, "FRAME_METRICS: %d frames of %dx%d (SSIM needs >= 11x11)", op.i0, op.H, op.W);
  MCVD_CHECK(op.B <= 65535, "FRAME_METRICS: batch %d too large for the grid", op.B);
  const size_t smem = (size_t)2 * op.H * op.W * sizeof(float);
  MCVD_CHECK(smem <= 200 * 1024, "FRAME_METRICS: %dx%d frames do not fit shared memory", op.H, op.W);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(k_frame_metrics, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    MCVD_CHECK(e == cudaSuccess, "FRAME_METRICS: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
  }
  dim3 grid(op.i0, op.B);
  k_frame_metrics<<<grid, 256, smem, s>>>((const float*)op.src0, (const float*)op.src1, (double*)op.dst, op.C0, op.i0,
                                          op.H, op.W, (op.flags & MCVD_F_ROUND) ? 1 : 0);
  MCVD_CUDA_LAUNCH_CHECK("frame_metrics");
  return 0;
}

}  // namespace mcvd
