// C-ABI entry points (include/mcvd_b200.h): program runner, validation, error reporting.
#include <stdarg.h>
#include <string.h>

#include "mcvd_common.cuh"

namespace mcvd {

static thread_local char g_err[512] = {0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static int dispatch(const McvdOp& op, cudaStream_t s) {
  switch (op.kind) {
    case MCVD_OP_NCHW_TO_NHWC: return launch_nchw_to_nhwc(op, s);
    case MCVD_OP_NHWC_TO_NCHW: return launch_nhwc_to_nchw(op, s);
    case MCVD_OP_TIMESTEP_EMBED: return launch_timestep_embed(op, s);
    case MCVD_OP_LINEAR: return launch_linear(op, s);
    case MCVD_OP_GN_PARTIAL: return launch_gn_partial(op, s);
    case MCVD_OP_GN_FINALIZE: return launch_gn_finalize(op, s);
    case MCVD_OP_APPLY: return launch_apply(op, s);
    case MCVD_OP_CONV_SIMT: return launch_conv_simt(op, s);
    case MCVD_OP_ATTENTION: return launch_attention(op, s);
    case MCVD_OP_RESIZE_NEAREST: return launch_resize_nearest(op, s);
    case MCVD_OP_DIFFUSION_UPDATE: return launch_diffusion_update(op, s);
    case MCVD_OP_CONV_UMMA: return launch_conv_umma(op, s);
    case MCVD_OP_CONV_UMMA2: return launch_conv_umma2(op, s);
    case MCVD_OP_CONV_SMALLN: return launch_conv_smalln(op, s);
    case MCVD_OP_COPY: return launch_copy(op, s);
    case MCVD_OP_ATTENTION_UMMA: return launch_attention_umma(op, s);
    case MCVD_OP_FRAME_METRICS: return launch_frame_metrics(op, s);
    default: break;
  }
  set_error("unknown op kind %d", op.kind);
  return -1;
}

static int validate_one(const McvdOp& op, int idx) {
  if (op.kind <= 0 || op.kind >= MCVD_OP__COUNT) {
    set_error("op %d: unknown kind %d", idx, op.kind);
    return -1;
  }
  if (op.B <= 0) {
    set_error("op %d (kind %d): batch %d", idx, op.kind, op.B);
    return -1;
  }
  const bool spatial = op.kind != MCVD_OP_TIMESTEP_EMBED && op.kind != MCVD_OP_LINEAR && op.kind != MCVD_OP_COPY;
  if (spatial && (op.H <= 0 || op.W <= 0)) {
    set_error("op %d (kind %d): spatial size %dx%d", idx, op.kind, op.H, op.W);
    return -1;
  }
  if (!op.src0 || !op.dst) {
    set_error("op %d (kind %d): null src0/dst", idx, op.kind);
    return -1;
  }
  if (op.C1 > 0 && !op.src1 && op.kind != MCVD_OP_DIFFUSION_UPDATE) {
    set_error("op %d (kind %d): C1=%d but src1 is null", idx, op.kind, op.C1);
    return -1;
  }
  auto misaligned = [](const void* p) { return p && (reinterpret_cast<uintptr_t>(p) & 15) != 0; };
  if (misaligned(op.src0) || misaligned(op.src1) || misaligned(op.dst) || misaligned(op.w) || misaligned(op.aux0) ||
      misaligned(op.aux1) || misaligned(op.aux2)) {
    set_error("op %d (kind %d): pointers must be 16-byte aligned", idx, op.kind);
    return -1;
  }
  switch (op.kind) {
    case MCVD_OP_APPLY:
      if (op.C0 % 4 || op.C1 % 4) {
        set_error("op %d APPLY: channels (%d,%d) not multiples of 4", idx, op.C0, op.C1);
        return -1;
      }
      break;
    case MCVD_OP_CONV_SIMT:
    case MCVD_OP_CONV_UMMA:
    case MCVD_OP_CONV_UMMA2:
      if (!op.w || (op.i0 != 1 && op.i0 != 3)) {
        set_error("op %d CONV: null weights or kernel size %d", idx, op.i0);
        return -1;
      }
      break;
    case MCVD_OP_ATTENTION:
    case MCVD_OP_ATTENTION_UMMA:
      if (op.i0 * op.i1 != op.C0) {
        set_error("op %d ATTENTION: heads %d x dim %d != %d", idx, op.i0, op.i1, op.C0);
        return -1;
      }
      if (op.kind == MCVD_OP_ATTENTION_UMMA && (!op.dst2 || (reinterpret_cast<uintptr_t>(op.dst2) & 15))) {
        set_error("op %d ATTENTION_UMMA: dst2 (operand-image scratch) is null or not 16-byte aligned", idx);
        return -1;
      }
      break;
    case MCVD_OP_NCHW_TO_NHWC:
      if ((op.flags & MCVD_F_NOISE) &&
          (!op.aux0 || !op.aux1 || op.i4 <= 0 || !((op.flags & MCVD_F_PHILOX) ? op.w : op.aux2) ||
           ((op.flags & MCVD_F_GAMMA) && !(op.flags & MCVD_F_PHILOX)))) {
        set_error("op %d NCHW_TO_NHWC: conditioning noise needs labels, schedule tables and a noise source "
                  "(buffer, or the Philox control block; Gamma noise is drawn in-kernel only)", idx);
        return -1;
      }
      break;
    case MCVD_OP_DIFFUSION_UPDATE:
      if ((op.flags & MCVD_F_GAMMA) && !(op.f6 >= 1.f && op.f7 > 0.f)) {
        set_error("op %d DIFFUSION_UPDATE: Gamma noise needs shape k >= 1 and scale theta > 0 (got %g, %g)", idx, op.f6,
                  op.f7);
        return -1;
      }
      break;
    default: break;
  }
  return 0;
}

}  // namespace mcvd

extern "C" {

int mcvd_abi_version(void) { return MCVD_ABI_VERSION; }
int mcvd_sizeof_op(void) { return (int)sizeof(McvdOp); }
const char* mcvd_last_error(void) { return mcvd::g_err; }

int mcvd_device_arch(void) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    cudaGetLastError();
    mcvd::set_error("no CUDA device");
    return -1;
  }
  cudaDeviceProp p;
  if (cudaGetDeviceProperties(&p, dev) != cudaSuccess) {
    cudaGetLastError();
    mcvd::set_error("cudaGetDeviceProperties failed");
    return -1;
  }
  return p.major * 10 + p.minor;
}

int mcvd_validate_program(const McvdOp* ops, int n) {
  if (!ops || n < 0) {
    mcvd::set_error("null program");
    return -1;
  }
  for (int i = 0; i < n; ++i) {
    int r = mcvd::validate_one(ops[i], i);
    if (r) return r;
  }
  return 0;
}

int mcvd_count_launches(const McvdOp* ops, int n) {
  if (!ops || n < 0) return -1;
  int total = 0;
  for (int i = 0; i < n; ++i) total += (ops[i].kind == MCVD_OP_ATTENTION_UMMA) ? 2 : 1;   // pre-split + attention
  return total;
}

int mcvd_run_program(const McvdOp* ops, int n, void* stream) {
  if (!ops || n < 0) {
    mcvd::set_error("null program");
    return -1;
  }
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  for (int i = 0; i < n; ++i) {
    int r = mcvd::dispatch(ops[i], s);
    if (r) {
      char tmp[400];
      strncpy(tmp, mcvd::g_err, sizeof(tmp) - 1);
      tmp[sizeof(tmp) - 1] = 0;
      mcvd::set_error("op %d (kind %d): %s", i, ops[i].kind, tmp);
      return r;
    }
  }
  return 0;
}

}  // extern "C"
