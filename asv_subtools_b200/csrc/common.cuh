// Shared host-side helpers: error reporting, launch counting, bf16 split helpers.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>
#include <mutex>

#include "../../include/xvb200.h"

namespace xvb {

// thread-local last error message (xvb_last_error)
void set_error(const char* fmt, ...);
// counts kernels launched by this library on this thread (xvb_extractor_last_launches)
extern thread_local long g_launches;

#define XVB_CHECK_ARG(cond, ...)        \
  do {                                  \
    if (!(cond)) {                      \
      ::xvb::set_error(__VA_ARGS__);    \
      return XVB_EINVAL;                \
    }                                   \
  } while (0)

#define XVB_CUDA(expr)                                                                         \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      ::xvb::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return XVB_ECUDA;                                                                        \
    }                                                                                          \
  } while (0)

#define XVB_LAUNCH_CHECK()                                                              \
  do {                                                                                  \
    ::xvb::g_launches++;                                                                \
    cudaError_t _e = cudaGetLastError();                                                \
    if (_e != cudaSuccess) {                                                            \
      ::xvb::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
      return XVB_ECUDA;                                                                 \
    }                                                                                   \
  } while (0)

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) applies to ONE device (context): opt in once per
// (kernel, device).  `done` is the call site's own bitset of device ordinals, so the first launch of a
// kernel on a second GPU of the same process opts in there too; thread-safe (a lost race sets it twice).
static inline int ensure_dyn_smem_impl(const void* kernel, int bytes, std::atomic<unsigned long long>& done) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) { set_error("cudaGetDevice failed: %s", cudaGetErrorString(e)); return XVB_ECUDA; }
  const unsigned long long bit = 1ull << (dev & 63);
  if (dev < 64 && (done.load(std::memory_order_acquire) & bit)) return XVB_OK;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(%d B dynamic smem) failed: %s", bytes, cudaGetErrorString(e)); return XVB_ECUDA; }
  if (dev < 64) done.fetch_or(bit, std::memory_order_release);
  return XVB_OK;
}
#define XVB_ENSURE_DYN_SMEM(kernel, bytes)                                                         \
  do {                                                                                             \
    static std::atomic<unsigned long long> _xvb_done{0};                                           \
    int _rc = ::xvb::ensure_dyn_smem_impl(reinterpret_cast<const void*>(kernel), (bytes), _xvb_done); \
    if (_rc) return _rc;                                                                           \
  } while (0)

int require_sm100();  // XVB_OK or XVB_ENODEVICE (cached per device)
int sm_count();

// fp32 -> (hi, lo) bf16 split: hi = rn(x), lo = rn(x - hi)
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}
__device__ __forceinline__ uint32_t pack_bf16x2(__nv_bfloat16 a, __nv_bfloat16 b) {
  return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b) << 16);
}

// Fused consumer of a score matrix (scoring.cu: xvb_trial_histogram): instead of storing
// S = A.B^T + row + col, every score is binned into a (2, nbins) histogram by trial class.
struct TrialHist {
  unsigned long long* hist;
  const int* row_label;
  const int* col_label;
  float lo, inv_w;
  int nbins;
  int symmetric;
  int unit_first, unit_stride;   // 256-row units walked by this launch: unit_first + k * unit_stride
};

// tdnn_gemm.cu: the tcgen05 layer behind xvb_tdnn_affine / xvb_tdnn_affine_ex.
int tdnn_affine_impl(const xvb_tdnn_args_t& args, void* stream, const TrialHist* hist = nullptr);

// Plan / launch split of the same layer (tdnn_gemm.cu): a GemmPlan freezes tile geometry, tensor maps, kernel
// instantiation and grid for one (shapes, pointers) combination; launching it costs one kernel launch (two for
// split-K).  `scratch`: gemm_plan_scratch_bytes() bytes that stay valid for the life of the plan (split-K partials).
struct GemmPlan;
size_t gemm_plan_scratch_bytes(const xvb_tdnn_args_t& args, const TrialHist* hist = nullptr);
int gemm_plan_build(GemmPlan** out, const xvb_tdnn_args_t& args, const TrialHist* hist, void* scratch);
int gemm_plan_launch(const GemmPlan* plan, void* stream, float* y_f32_override = nullptr);
void gemm_plan_destroy(GemmPlan* plan);

// pooling.cu: launch of the fused-pooling merge behind xvb_pool_finalize; lengths (B, device) or NULL (all T frames)
int pool_finalize_launch(const float* partial, int num_blocks, int frames_per_block, int B, int T, int C, float eps, int mode,
                         const int32_t* lengths, float* out, uint16_t* out_hi, uint16_t* out_lo, int64_t ldo, void* stream);

// core.cu: ragged (sum_T, C) fp32 frames, utterance b = rows offsets[b] .. offsets[b+1] (device int32), -> split planes
// (B, pad_front + Tq + pad_back, ldp) with zero frames outside [0, L_b) of every utterance
int split_ragged_frames(const float* x, const int32_t* offsets, int B, int Tq, int C, uint16_t* hi, uint16_t* lo, int64_t ldp,
                        int pad_front, int pad_back, void* stream);

// tdnn_gemm.cu: cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda).
int make_tensor_map(CUtensorMap* m, const void* base, int esize, int rank, const unsigned long long* dims,
                    const unsigned long long* strides_bytes, const unsigned* box, int swizzle_bytes);

// stream-ordered scratch from the device's default memory pool
struct TempBuf {
  void* p = nullptr;
  cudaStream_t s;
  explicit TempBuf(cudaStream_t st) : s(st) {}
  int alloc(size_t bytes) {
    // keep freed scratch in the device's pool: with the default release threshold (0) every
    // synchronisation hands it back to the driver and the next call pays for mapping it again
    static std::once_flag once[64];
    int dev = 0;
    XVB_CUDA(cudaGetDevice(&dev));
    std::call_once(once[dev & 63], [dev] {
      cudaMemPool_t pool;
      if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        unsigned long long keep = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
      }
    });
    XVB_CUDA(cudaMallocAsync(&p, bytes, s));
    return XVB_OK;
  }
  ~TempBuf() { if (p) cudaFreeAsync(p, s); }
};

static inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

}  // namespace xvb
