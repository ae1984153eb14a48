// Statistics pooling over time (StatisticsPooling.forward, pytorch/libs/nnet/pooling.py:58-67).
//
//   mean[b,c] = (1/T) sum_t x[b,t,c];  std[b,c] = sqrt(max((1/T) sum_t (x-mean)^2, eps))
//
// HBM-bound: x (B,T,C) fp32 is read exactly once.  A CTA owns one utterance x one 128-channel
// slab.  The slab (up to 200 frames x 512 B = 100 KB) is pulled into shared memory by TMA in
// 40-frame boxes, each with its own mbarrier, so ~100 KB per CTA (two CTAs per SM) are in flight
// without costing registers, and the reduction starts on the first box while the rest lands.
// With the slab on chip the statistics are the reference's literal two passes: pass 1 the mean,
// pass 2 sum((x - mean)^2).  Utterances longer than one slab are processed slab by slab and merged
// with Chan's parallel-variance update (algebraically the same two-pass result).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "common.cuh"
#include "ptx.cuh"

namespace xvb {

constexpr int kPoolWarps = 8;
constexpr int kPoolBoxRows = 40;                 // frames per TMA box (20 KB)
constexpr int kPoolSlabRows = 200;               // 5 boxes resident: 100 KB -> two CTAs per SM
constexpr int kPoolNumBars = (kPoolSlabRows + kPoolBoxRows - 1) / kPoolBoxRows;
constexpr int kPoolSmemBytes = kPoolNumBars * kPoolBoxRows * 128 * 4 + kPoolWarps * 128 * 4 + 128 + 128 /* alignment slack */;

__global__ void __launch_bounds__(kPoolWarps * 32, 2)
stats_pool_tma_kernel(const __grid_constant__ CUtensorMap map_x, int T, int C, float eps, int mode, float* __restrict__ out,
                      __nv_bfloat16* __restrict__ out_hi, __nv_bfloat16* __restrict__ out_lo, long long ldo) {
  // TMA destinations need 128-byte alignment; CUDA only promises 16 for dynamic shared memory (and a tool that adds
  // its own static shared memory, e.g. compute-sanitizer, does shift the base), so align by hand
  extern __shared__ uint8_t pool_smem_raw[];
  uint8_t* pool_smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(pool_smem_raw) + 127) & ~uintptr_t(127));
  float* slab = reinterpret_cast<float*>(pool_smem);                                  // [rows][128]
  float* scratch = slab + kPoolNumBars * kPoolBoxRows * 128;                          // [warps][128]
  uint64_t* bars = reinterpret_cast<uint64_t*>(scratch + kPoolWarps * 128);           // [kPoolNumBars]

  const int b = blockIdx.y;
  const int c0 = blockIdx.x * 128;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = c0 + lane * 4;
  const bool active = c < C;  // C % 4 == 0

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&map_x);
    for (int i = 0; i < kPoolNumBars; ++i) mbar_init(&bars[i], 1);
    fence_barrier_init();
  }
  __syncthreads();

  float run_n = 0.f;
  float4 run_mean = make_float4(0.f, 0.f, 0.f, 0.f), run_m2 = make_float4(0.f, 0.f, 0.f, 0.f);
  uint32_t phase = 0;
  for (int t_base = 0; t_base < T; t_base += kPoolSlabRows, phase ^= 1) {
    const int rows = min(kPoolSlabRows, T - t_base);
    const int nbox = (rows + kPoolBoxRows - 1) / kPoolBoxRows;
    if (threadIdx.x == 0) {
      for (int i = 0; i < nbox; ++i) {
        mbar_expect_tx(&bars[i], kPoolBoxRows * 128 * 4);  // OOB rows/channels are zero-filled but counted
        tma_load_3d(slab + i * kPoolBoxRows * 128, &map_x, &bars[i], c0, t_base + i * kPoolBoxRows, b);
      }
    }
    // ---- pass 1: mean (rows strided over warps; start as soon as a box has landed)
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i = 0; i < nbox; ++i) {
      mbar_wait(&bars[i], phase);
      const int r_end = min(rows, (i + 1) * kPoolBoxRows);
#pragma unroll 4
      for (int r = i * kPoolBoxRows + warp; r < r_end; r += kPoolWarps) {
        const float4 v = *reinterpret_cast<const float4*>(slab + r * 128 + lane * 4);
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
      }
    }
    *reinterpret_cast<float4*>(scratch + warp * 128 + lane * 4) = s;
    __syncthreads();
    float4 m = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int w = 0; w < kPoolWarps; ++w) {
      const float4 v = *reinterpret_cast<const float4*>(scratch + w * 128 + lane * 4);
      m.x += v.x; m.y += v.y; m.z += v.z; m.w += v.w;
    }
    const float inv = 1.f / (float)rows;
    m.x *= inv; m.y *= inv; m.z *= inv; m.w *= inv;
    __syncthreads();
    // ---- pass 2: sum (x - mean)^2 from the on-chip slab
    float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
    for (int r = warp; r < rows; r += kPoolWarps) {
      const float4 v = *reinterpret_cast<const float4*>(slab + r * 128 + lane * 4);
      float d;
      d = v.x - m.x; q.x = fmaf(d, d, q.x);
      d = v.y - m.y; q.y = fmaf(d, d, q.y);
      d = v.z - m.z; q.z = fmaf(d, d, q.z);
      d = v.w - m.w; q.w = fmaf(d, d, q.w);
    }
    *reinterpret_cast<float4*>(scratch + warp * 128 + lane * 4) = q;
    __syncthreads();
    float4 m2 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int w = 0; w < kPoolWarps; ++w) {
      const float4 v = *reinterpret_cast<const float4*>(scratch + w * 128 + lane * 4);
      m2.x += v.x; m2.y += v.y; m2.z += v.z; m2.w += v.w;
    }
    __syncthreads();  // scratch and slab are free again
    // ---- Chan merge of this slab into the running statistics (every thread keeps a copy)
    const float nb = (float)rows, tot = run_n + nb, wb = nb / tot, cross = run_n * wb;
    float d;
    d = m.x - run_mean.x; run_mean.x = fmaf(d, wb, run_mean.x); run_m2.x += m2.x + d * d * cross;
    d = m.y - run_mean.y; run_mean.y = fmaf(d, wb, run_mean.y); run_m2.y += m2.y + d * d * cross;
    d = m.z - run_mean.z; run_mean.z = fmaf(d, wb, run_mean.z); run_m2.z += m2.z + d * d * cross;
    d = m.w - run_mean.w; run_mean.w = fmaf(d, wb, run_mean.w); run_m2.w += m2.w + d * d * cross;
    run_n = tot;
  }

  if (warp == 0 && active) {
    float sd[4];
    if (mode == 0) {  // StatisticsPooling: sqrt(clamp(biased var, eps))  (pooling.py:62-66)
      const float invT = 1.f / (float)T;
      sd[0] = sqrtf(fmaxf(run_m2.x * invT, eps)); sd[1] = sqrtf(fmaxf(run_m2.y * invT, eps));
      sd[2] = sqrtf(fmaxf(run_m2.z * invT, eps)); sd[3] = sqrtf(fmaxf(run_m2.w * invT, eps));
    } else {          // ECAPA global context: sqrt(unbiased var + eps)  (ecapa_tdnn_xvector.py:177-178; T=1 -> NaN as there)
      const float invT1 = 1.f / (float)(T - 1);
      sd[0] = sqrtf(run_m2.x * invT1 + eps); sd[1] = sqrtf(run_m2.y * invT1 + eps);
      sd[2] = sqrtf(run_m2.z * invT1 + eps); sd[3] = sqrtf(run_m2.w * invT1 + eps);
    }
    float mu[4] = {run_mean.x, run_mean.y, run_mean.z, run_mean.w};
    float* ob = out + (long long)b * 2 * C;
    *reinterpret_cast<float4*>(ob + c) = make_float4(mu[0], mu[1], mu[2], mu[3]);
    *reinterpret_cast<float4*>(ob + C + c) = make_float4(sd[0], sd[1], sd[2], sd[3]);
    if (out_hi) {
      __nv_bfloat16 h[8], l[8];
#pragma unroll
      for (int k = 0; k < 4; ++k) { split_bf16(mu[k], h[k], l[k]); split_bf16(sd[k], h[4 + k], l[4 + k]); }
      __nv_bfloat16* oh = out_hi + (long long)b * ldo;
      __nv_bfloat16* ol = out_lo + (long long)b * ldo;
      *reinterpret_cast<uint2*>(oh + c) = make_uint2(pack_bf16x2(h[0], h[1]), pack_bf16x2(h[2], h[3]));
      *reinterpret_cast<uint2*>(ol + c) = make_uint2(pack_bf16x2(l[0], l[1]), pack_bf16x2(l[2], l[3]));
      *reinterpret_cast<uint2*>(oh + C + c) = make_uint2(pack_bf16x2(h[4], h[5]), pack_bf16x2(h[6], h[7]));
      *reinterpret_cast<uint2*>(ol + C + c) = make_uint2(pack_bf16x2(l[4], l[5]), pack_bf16x2(l[6], l[7]));
    }
  }
}

// Merge the per-time-block [mean | M2] partials written by the fused GEMM epilogue (Chan's update,
// block k has n_k = min(Tb, T - k*Tb) frames), then apply the reference's std definition.  Ragged batch
// (lengths != NULL): utterance b has L = lengths[b] frames, so only its first ceil(L / Tb) blocks were
// written -- the rest are never read -- and L is the divisor.
__global__ void pool_finalize_kernel(const float* __restrict__ partial, int nblk, int Tb, int B, int T, int C, float eps,
                                     int mode, const int* __restrict__ lengths, float* __restrict__ out,
                                     __nv_bfloat16* __restrict__ out_hi, __nv_bfloat16* __restrict__ out_lo, long long ldo) {
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  const int b = blockIdx.y;
  if (c >= C) return;
  if (lengths) {
    T = min(lengths[b], T);
    nblk = min(nblk, (T + Tb - 1) / Tb);
  }
  float n = 0.f;
  float mean[4] = {0.f, 0.f, 0.f, 0.f}, m2[4] = {0.f, 0.f, 0.f, 0.f};
  for (int k = 0; k < nblk; ++k) {
    const float* p = partial + ((long long)k * B + b) * (2LL * C) + c;
    const float4 mk = *reinterpret_cast<const float4*>(p);
    const float4 qk = *reinterpret_cast<const float4*>(p + C);
    const float nk = (float)min(Tb, T - k * Tb), tot = n + nk, wb = nk / tot, cross = n * wb;
    const float mv[4] = {mk.x, mk.y, mk.z, mk.w}, qv[4] = {qk.x, qk.y, qk.z, qk.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float d = mv[j] - mean[j];
      mean[j] = fmaf(d, wb, mean[j]);
      m2[j] += qv[j] + d * d * cross;
    }
    n = tot;
  }
  float sd[4];
#pragma unroll
  for (int j = 0; j < 4; ++j)
    sd[j] = mode == 0 ? sqrtf(fmaxf(m2[j] / (float)T, eps)) : sqrtf(m2[j] / (float)(T - 1) + eps);
  float* ob = out + (long long)b * 2 * C;
  *reinterpret_cast<float4*>(ob + c) = make_float4(mean[0], mean[1], mean[2], mean[3]);
  *reinterpret_cast<float4*>(ob + C + c) = make_float4(sd[0], sd[1], sd[2], sd[3]);
  if (out_hi) {
    __nv_bfloat16 h[8], l[8];
#pragma unroll
    for (int k = 0; k < 4; ++k) { split_bf16(mean[k], h[k], l[k]); split_bf16(sd[k], h[4 + k], l[4 + k]); }
    __nv_bfloat16* oh = out_hi + (long long)b * ldo;
    __nv_bfloat16* ol = out_lo + (long long)b * ldo;
    *reinterpret_cast<uint2*>(oh + c) = make_uint2(pack_bf16x2(h[0], h[1]), pack_bf16x2(h[2], h[3]));
    *reinterpret_cast<uint2*>(ol + c) = make_uint2(pack_bf16x2(l[0], l[1]), pack_bf16x2(l[2], l[3]));
    *reinterpret_cast<uint2*>(oh + C + c) = make_uint2(pack_bf16x2(h[4], h[5]), pack_bf16x2(h[6], h[7]));
    *reinterpret_cast<uint2*>(ol + C + c) = make_uint2(pack_bf16x2(l[4], l[5]), pack_bf16x2(l[6], l[7]));
  }
}

int pool_finalize_launch(const float* partial, int num_blocks, int frames_per_block, int B, int T, int C, float eps, int mode,
                         const int32_t* lengths, float* out, uint16_t* out_hi, uint16_t* out_lo, int64_t ldo, void* stream) {
  dim3 grid((C / 4 + 127) / 128, B);
  pool_finalize_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(partial, num_blocks, frames_per_block, B, T, C, eps, mode, lengths,
                                                              out, reinterpret_cast<__nv_bfloat16*>(out_hi),
                                                              reinterpret_cast<__nv_bfloat16*>(out_lo), ldo);
  XVB_LAUNCH_CHECK();
  return XVB_OK;
}

}  // namespace xvb

using namespace xvb;

extern "C" int xvb_pool_finalize(const float* partial, int num_blocks, int frames_per_block, int B, int T, int C, float eps,
                                 int mode, float* out, uint16_t* out_hi, uint16_t* out_lo, int64_t ldo, void* stream) {
  int rc = require_sm100();
  if (rc) return rc;
  XVB_CHECK_ARG(partial && out && num_blocks > 0 && frames_per_block > 0 && B > 0 && T > 0 && C > 0 && C % 4 == 0 && B <= 65535,
                "xvb_pool_finalize: bad arguments");
  XVB_CHECK_ARG((long long)num_blocks * frames_per_block >= T && (long long)(num_blocks - 1) * frames_per_block < T,
                "xvb_pool_finalize: %d blocks of %d frames do not tile T=%d", num_blocks, frames_per_block, T);
  XVB_CHECK_ARG((out_hi != nullptr) == (out_lo != nullptr), "xvb_pool_finalize: out_hi/out_lo must both be set or both NULL");
  if (out_hi) XVB_CHECK_ARG(ldo >= 2 * C && ldo % 4 == 0, "xvb_pool_finalize: ldo too small / unaligned");
  XVB_CHECK_ARG(mode == 0 || mode == 1, "xvb_pool_finalize: mode must be 0 or 1");
  return pool_finalize_launch(partial, num_blocks, frames_per_block, B, T, C, eps, mode, nullptr, out, out_hi, out_lo, ldo, stream);
}

extern "C" int xvb_stats_pool(const float* x, int64_t ldx, int B, int T, int C, float eps, float* out, uint16_t* out_hi,
                              uint16_t* out_lo, int64_t ldo, void* stream) {
  return xvb_stats_pool_ex(x, ldx, B, T, C, eps, 0, out, out_hi, out_lo, ldo, stream);
}

extern "C" int xvb_stats_pool_ex(const float* x, int64_t ldx, int B, int T, int C, float eps, int mode, float* out,
                                 uint16_t* out_hi, uint16_t* out_lo, int64_t ldo, void* stream) {
  int rc = require_sm100();
  if (rc) return rc;
  XVB_CHECK_ARG(x && out, "xvb_stats_pool: null pointer");
  XVB_CHECK_ARG(mode == 0 || mode == 1, "xvb_stats_pool_ex: mode must be 0 (biased, clamp) or 1 (unbiased, +eps)");
  XVB_CHECK_ARG(B > 0 && T > 0 && C > 0 && C % 4 == 0 && ldx % 4 == 0 && ldx >= C, "xvb_stats_pool: need C%%4==0, ldx%%4==0 (C=%d ldx=%lld)", C, (long long)ldx);
  XVB_CHECK_ARG((out_hi != nullptr) == (out_lo != nullptr), "xvb_stats_pool: out_hi/out_lo must both be set or both NULL");
  if (out_hi) XVB_CHECK_ARG(ldo >= 2 * C && ldo % 4 == 0, "xvb_stats_pool: ldo=%lld too small / unaligned", (long long)ldo);
  XVB_CHECK_ARG(((uintptr_t)x | (uintptr_t)out) % 16 == 0 && ((uintptr_t)out_hi | (uintptr_t)out_lo) % 8 == 0, "xvb_stats_pool: unaligned pointer");
  XVB_CHECK_ARG(B <= 65535, "xvb_stats_pool: B=%d exceeds grid.y", B);
  CUtensorMap map;
  const unsigned long long dims[3] = {(unsigned long long)C, (unsigned long long)T, (unsigned long long)B};
  const unsigned long long strides[2] = {(unsigned long long)ldx * 4, (unsigned long long)ldx * 4 * (unsigned long long)T};
  const unsigned box[3] = {128u, (unsigned)kPoolBoxRows, 1u};
  rc = make_tensor_map(&map, x, 4, 3, dims, strides, box, 0);
  if (rc) return rc;
  XVB_ENSURE_DYN_SMEM((stats_pool_tma_kernel), kPoolSmemBytes);
  dim3 grid((C + 127) / 128, B);
  stats_pool_tma_kernel<<<grid, kPoolWarps * 32, kPoolSmemBytes, (cudaStream_t)stream>>>(
      map, T, C, eps, mode, out, reinterpret_cast<__nv_bfloat16*>(out_hi), reinterpret_cast<__nv_bfloat16*>(out_lo), ldo);
  XVB_LAUNCH_CHECK();
  return XVB_OK;
}
