// Library core: error reporting, device check, frame-matrix staging, weight packing, the SIMT
// cross-check layer.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <string.h>

#include "common.cuh"

namespace xvb {

static thread_local char g_err[512] = "";
thread_local long g_launches = 0;

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int require_sm100() {
  static thread_local int cached_dev = -1;
  static thread_local int cached_rc = XVB_ENODEVICE;
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    cudaGetLastError();
    set_error("no CUDA device visible: libxvb200 has no CPU fallback");
    return XVB_ENODEVICE;
  }
  if (dev == cached_dev) {
    if (cached_rc) set_error("device %d is not sm_100 (B200): libxvb200 has no fallback path", dev);
    return cached_rc;
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) {
    cudaGetLastError();
    set_error("cudaGetDeviceProperties failed");
    return XVB_ENODEVICE;
  }
  cached_dev = dev;
  cached_rc = (prop.major == 10) ? XVB_OK : XVB_ENODEVICE;
  if (cached_rc) set_error("device %d is sm_%d%d, need sm_100 (B200): libxvb200 has no fallback path", dev, prop.major, prop.minor);
  return cached_rc;
}

int sm_count() {
  static thread_local int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

// ------------------------------------------------------------------------------------------------
// fp32 rows -> split planes.  One thread per 8 output columns (16-byte stores).
// ------------------------------------------------------------------------------------------------
__global__ void split_f32_kernel(const float* __restrict__ x, long long rows, int C, long long ldx,
                                 __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo, long long ldp) {
  const long long groups_per_row = ldp / 8;
  const long long total = rows * groups_per_row;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / groups_per_row;
    const int c0 = (int)(i % groups_per_row) * 8;
    uint32_t h[4], l[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int c = c0 + 2 * k;
      const float a = c < C ? x[r * ldx + c] : 0.f;
      const float b = c + 1 < C ? x[r * ldx + c + 1] : 0.f;
      __nv_bfloat16 ah, al, bh, bl;
      split_bf16(a, ah, al);
      split_bf16(b, bh, bl);
      h[k] = pack_bf16x2(ah, bh);
      l[k] = pack_bf16x2(al, bl);
    }
    *reinterpret_cast<uint4*>(hi + r * ldp + c0) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(lo + r * ldp + c0) = make_uint4(l[0], l[1], l[2], l[3]);
  }
}

// (B, T, C) fp32 frames -> planes (B, pad_front + T + pad_back, ldp) with zero frames around each
// utterance.  One thread per 8 output columns; float4 loads when the source rows allow it.
__global__ void split_frames_kernel(const float* __restrict__ x, int B, int T, int C, __nv_bfloat16* __restrict__ hi,
                                    __nv_bfloat16* __restrict__ lo, long long ldp, int pad_front, int Tp, int vec) {
  const long long groups_per_row = ldp / 8;
  const long long total = (long long)B * Tp * groups_per_row;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / groups_per_row;
    const int c0 = (int)(i - r * groups_per_row) * 8;
    const int b = (int)(r / Tp), t = (int)(r - (long long)b * Tp) - pad_front;
    float v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = 0.f;
    if (t >= 0 && t < T) {
      const float* src = x + ((long long)b * T + t) * C + c0;
      if (vec && c0 + 8 <= C) {
        const float4 a = *reinterpret_cast<const float4*>(src), c = *reinterpret_cast<const float4*>(src + 4);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = c.x; v[5] = c.y; v[6] = c.z; v[7] = c.w;
      } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) if (c0 + k < C) v[k] = src[k];
      }
    }
    uint32_t h[4], l[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      __nv_bfloat16 ah, al, bh, bl;
      split_bf16(v[2 * k], ah, al);
      split_bf16(v[2 * k + 1], bh, bl);
      h[k] = pack_bf16x2(ah, bh);
      l[k] = pack_bf16x2(al, bl);
    }
    *reinterpret_cast<uint4*>(hi + r * ldp + c0) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(lo + r * ldp + c0) = make_uint4(l[0], l[1], l[2], l[3]);
  }
}

// The same from a ragged batch: utterance b is rows offsets[b] .. offsets[b+1] of x (sum_T, C) and is
// padded with zero frames up to Tq (so time steps [L_b, Tq) read as F.pad zeros, like the reference's
// one-utterance extraction).
__global__ void split_ragged_kernel(const float* __restrict__ x, const int32_t* __restrict__ offsets, int C,
                                    __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo, long long ldp,
                                    int pad_front, int Tp, long long total, int vec) {
  const long long groups_per_row = ldp / 8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / groups_per_row;
    const int c0 = (int)(i - r * groups_per_row) * 8;
    const int b = (int)(r / Tp), t = (int)(r - (long long)b * Tp) - pad_front;
    const int row0 = offsets[b], len = offsets[b + 1] - row0;
    float v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = 0.f;
    if (t >= 0 && t < len) {
      const float* src = x + ((long long)row0 + t) * C + c0;
      if (vec && c0 + 8 <= C) {
        const float4 a = *reinterpret_cast<const float4*>(src), c = *reinterpret_cast<const float4*>(src + 4);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = c.x; v[5] = c.y; v[6] = c.z; v[7] = c.w;
      } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) if (c0 + k < C) v[k] = src[k];
      }
    }
    uint32_t h[4], l[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      __nv_bfloat16 ah, al, bh, bl;
      split_bf16(v[2 * k], ah, al);
      split_bf16(v[2 * k + 1], bh, bl);
      h[k] = pack_bf16x2(ah, bh);
      l[k] = pack_bf16x2(al, bl);
    }
    *reinterpret_cast<uint4*>(hi + r * ldp + c0) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(lo + r * ldp + c0) = make_uint4(l[0], l[1], l[2], l[3]);
  }
}

// ------------------------------------------------------------------------------------------------
// Reference weight (Cout, Cin, tot) -> packed K-major planes (Cout, ntaps*cin_p16), masked taps dropped.
// ------------------------------------------------------------------------------------------------
struct PackCtx { int ctx[XVB_MAX_TAPS]; };

__global__ void pack_weight_kernel(const float* __restrict__ w, int Cout, int Cin, int tot, int left, PackCtx pc,
                                   int ntaps, int cin_p16, __nv_bfloat16* __restrict__ whi,
                                   __nv_bfloat16* __restrict__ wlo) {
  const long long K = (long long)ntaps * cin_p16;
  const long long total = (long long)Cout * K;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(i / K);
    const int k = (int)(i % K);
    const int tap = k / cin_p16, c = k % cin_p16;
    float v = 0.f;
    if (c < Cin) v = w[((long long)n * Cin + c) * tot + (pc.ctx[tap] - left)];
    __nv_bfloat16 h, l;
    split_bf16(v, h, l);
    whi[i] = h;
    wlo[i] = l;
  }
}

// ------------------------------------------------------------------------------------------------
// SIMT fp32 cross-check layer: one thread per (frame, n); reads the unpacked reference weight.
// ------------------------------------------------------------------------------------------------
__global__ void tdnn_simt_kernel(const float* __restrict__ x, long long ldx, const float* __restrict__ w, int tot,
                                 int left, const float* __restrict__ bias, const float* __restrict__ scale,
                                 const float* __restrict__ shift, int flags, PackCtx pc, int ntaps,
                                 float* __restrict__ y, long long ldy, int B, int T, int Cin, int Cout) {
  const long long total = (long long)B * T * Cout;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(i % Cout);
    const long long frame = i / Cout;
    const int t = (int)(frame % T);
    const long long b = frame / T;
    float acc = bias ? bias[n] : 0.f;
    for (int tap = 0; tap < ntaps; ++tap) {
      const int tt = t + pc.ctx[tap];
      if (tt < 0 || tt >= T) continue;  // F.pad zeros (components.py:117)
      const float* xr = x + (b * T + tt) * ldx;
      const float* wr = w + (long long)n * Cin * tot + (pc.ctx[tap] - left);
      float s = 0.f;
      for (int c = 0; c < Cin; ++c) s = fmaf(xr[c], wr[(long long)c * tot], s);
      acc += s;
    }
    if (flags & XVB_RELU) acc = fmaxf(acc, 0.f);
    if (flags & XVB_BN) acc = fmaf(acc, scale[n], shift[n]);
    y[frame * ldy + n] = acc;
  }
}

static int grid_for(long long total, int block) {
  long long g = (total + block - 1) / block;
  const long long cap = (long long)sm_count() * 16;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

int split_ragged_frames(const float* x, const int32_t* offsets, int B, int Tq, int C, uint16_t* hi, uint16_t* lo, int64_t ldp,
                        int pad_front, int pad_back, void* stream) {
  XVB_CHECK_ARG(x && offsets && hi && lo && B > 0 && Tq > 0 && C > 0 && ldp >= C && ldp % 8 == 0 && pad_front >= 0 && pad_back >= 0,
                "split_ragged_frames: bad arguments");
  const int Tp = pad_front + Tq + pad_back;
  const long long total = (long long)B * Tp * (ldp / 8);
  const int vec = (C % 4 == 0 && (uintptr_t)x % 16 == 0) ? 1 : 0;
  split_ragged_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
      x, offsets, C, reinterpret_cast<__nv_bfloat16*>(hi), reinterpret_cast<__nv_bfloat16*>(lo), ldp, pad_front, Tp, total, vec);
  XVB_LAUNCH_CHECK();
  return XVB_OK;
}

}  // namespace xvb

using namespace xvb;

extern "C" int xvb_version(void) { return XVB_VERSION; }
extern "C" const char* xvb_last_error(void) { return g_err; }
extern "C" int xvb_device_check(void) { return require_sm100(); }

extern "C" int xvb_split_f32(const float* x, int64_t rows, int C, int64_t ldx, uint16_t* hi, uint16_t* lo, int64_t ldp,
                             void* stream) {
  int rc = require_sm100();
  if (rc) return rc;
  XVB_CHECK_ARG(x && hi && lo, "xvb_split_f32: null pointer");
  XVB_CHECK_ARG(rows > 0 && C > 0 && ldx >= C && ldp >= C && ldp % 8 == 0, "xvb_split_f32: bad shape rows=%lld C=%d ldx=%lld ldp=%lld",
                (long long)rows, C, (long long)ldx, (long long)ldp);
  XVB_CHECK_ARG(((uintptr_t)hi | (uintptr_t)lo) % 16 == 0, "xvb_split_f32: planes must be 16-byte aligned");
  const long long total = rows * (ldp / 8);
  split_f32_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
      x, rows, C, ldx, reinterpret_cast<__nv_bfloat16*>(hi), reinterpret_cast<__nv_bfloat16*>(lo), ldp);
  XVB_LAUNCH_CHECK();
  return XVB_OK;
}

extern "C" int xvb_split_frames(const float* x, int B, int T, int C, uint16_t* hi, uint16_t* lo, int64_t ldp, int pad_front,
                                int pad_back, void* stream) {
  int rc = require_sm100();
  if (rc) return rc;
  XVB_CHECK_ARG(x && hi && lo && B > 0 && T > 0 && C > 0 && ldp >= C && ldp % 8 == 0 && pad_front >= 0 && pad_back >= 0,
                "xvb_split_frames: bad arguments");
  XVB_CHECK_ARG(((uintptr_t)hi | (uintptr_t)lo) % 16 == 0, "xvb_split_frames: planes must be 16-byte aligned");
  const int Tp = pad_front + T + pad_back;
  const long long total = (long long)B * Tp * (ldp / 8);
  const int vec = (C % 4 == 0 && (uintptr_t)x % 16 == 0) ? 1 : 0;
  split_frames_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
      x, B, T, C, reinterpret_cast<__nv_bfloat16*>(hi), reinterpret_cast<__nv_bfloat16*>(lo), ldp, pad_front, Tp, vec);
  XVB_LAUNCH_CHECK();
  return XVB_OK;
}

extern "C" int64_t xvb_packed_weight_elems(int Cout, int Cin, int ntaps) {
  return (int64_t)Cout * ntaps * round_up(Cin, 16);
}

extern "C" int xvb_pack_tdnn_weight(const float* w, int Cout, int Cin, int tot_context, int left_context,
                                    const int* context_host, int ntaps, uint16_t* w_hi, uint16_t* w_lo, void* stream) {
  int rc = require_sm100();
  if (rc) return rc;
  XVB_CHECK_ARG(w && w_hi && w_lo && context_host, "xvb_pack_tdnn_weight: null pointer");
  XVB_CHECK_ARG(ntaps >= 1 && ntaps <= XVB_MAX_TAPS, "xvb_pack_tdnn_weight: ntaps=%d out of range", ntaps);
  PackCtx pc{};
  for (int i = 0; i < ntaps; ++i) {
    const int off = context_host[i] - left_context;
    XVB_CHECK_ARG(off >= 0 && off < tot_context, "xvb_pack_tdnn_weight: context %d outside the stored kernel [%d,%d)",
                  context_host[i], left_context, left_context + tot_context);
    pc.ctx[i] = context_host[i];
  }
  const int cin_p16 = (int)round_up(Cin, 16);
  const long long total = (long long)Cout * ntaps * cin_p16;
  pack_weight_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
      w, Cout, Cin, tot_context, left_context, pc, ntaps, cin_p16, reinterpret_cast<__nv_bfloat16*>(w_hi),
      reinterpret_cast<__nv_bfloat16*>(w_lo));
  XVB_LAUNCH_CHECK();
  return XVB_OK;
}

extern "C" int xvb_tdnn_affine_simt(const float* x, int64_t ldx, const float* w, int tot_context, int left_context,
                                    const float* bias, const float* bn_scale, const float* bn_shift, int flags,
                                    const int* context_host, int ntaps, float* y, int64_t ldy, int B, int T, int Cin,
                                    int Cout, void* stream) {
  int rc = require_sm100();
  if (rc) return rc;
  XVB_CHECK_ARG(x && w && y && context_host, "xvb_tdnn_affine_simt: null pointer");
  XVB_CHECK_ARG(ntaps >= 1 && ntaps <= XVB_MAX_TAPS, "xvb_tdnn_affine_simt: ntaps=%d out of range", ntaps);
  XVB_CHECK_ARG(!(flags & XVB_BN) || (bn_scale && bn_shift), "xvb_tdnn_affine_simt: XVB_BN without scale/shift");
  PackCtx pc{};
  for (int i = 0; i < ntaps; ++i) {
    const int off = context_host[i] - left_context;
    XVB_CHECK_ARG(off >= 0 && off < tot_context, "xvb_tdnn_affine_simt: context outside the stored kernel");
    pc.ctx[i] = context_host[i];
  }
  const long long total = (long long)B * T * Cout;
  tdnn_simt_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
      x, ldx, w, tot_context, left_context, bias, bn_scale, bn_shift, flags, pc, ntaps, y, ldy, B, T, Cin, Cout);
  XVB_LAUNCH_CHECK();
  return XVB_OK;
}
