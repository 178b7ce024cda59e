// common.cuh — context, error plumbing and small device helpers shared by all TUs
// of libmpn_b200.so. sm_100a only.
#pragma once
#include <utility>
#include <stdlib.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>
#include "../../include/mpn_abi.h"

struct mpn_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  int sm_count = 148;
  std::string err;
  int64_t launches = 0;
  // scratch owned by the ctx (grown on demand, never shrunk)
  void *scratch = nullptr; size_t scratch_bytes = 0;
  void *scratch2 = nullptr; size_t scratch2_bytes = 0;
  void *scratch3 = nullptr; size_t scratch3_bytes = 0;   // split-K partial accumulators
  void *small_dev = nullptr;                               // 256 bytes for scalar reductions (mpn_absmax)
  // optional per-category kernel timing (bench.py roofline): CUDA events around every launch group
  int profiling = 0;
  struct ProfRec { int cat; cudaEvent_t a, b; };
  std::vector<ProfRec> prof;
  std::vector<cudaEvent_t> ev_pool;
  uint8_t tc_attr_set[32] = {0};
  // stream-K (gemm_tc.cu): per-CTA partial-tile slots + per-(CTA, epilogue warp) flags holding the launch epoch
  float *sk_ws = nullptr; unsigned *sk_flags = nullptr; unsigned sk_epoch = 0;
  // NMS tie flags live in scratch2 and are reset by their last reader; (pointer, count) of the region known to be zero
  void *nms_tie_ptr = nullptr; int nms_tie_n = 0;
  // in-kernel timeline of the tcgen05 launches (diagnostics, mpn_ctx_timeline_begin/end): per launch 4 min- and 4 max-stamps
  unsigned long long *tl_min = nullptr, *tl_max = nullptr; int tl_cap = 0, tl_n = 0, tl_on = 0;
  // the end-of-run all-gather (dist.cu): an ncclComm_t bound at run time, this ctx's rank / world, collectives issued
  // run-time knobs (mpn_ctx_set_option); -1 = take the environment default
  int opt_roi_norm_split = -1, opt_roi_impl = -1, opt_fc_w16 = -1;
  // fp16 activation planes (fc6 / fc7 "w16" numerics): a value beyond fp16's range saturates AND raises this device flag;
  // host-synchronous entry points copy it to the pinned word with their results and fail loudly (mpn_check_overflow)
  unsigned *ovf_dev = nullptr; unsigned *ovf_host = nullptr;
  void *dist_comm = nullptr; int dist_rank = 0, dist_world = 1; int64_t collectives = 0;
  int own_stream = 0;              // mpn_ctx_create_stream: the ctx created (and destroys) its stream
  cudaEvent_t join_ev = nullptr;   // mpn_ctx_wait_ctx
  float *u8_lut_dev = nullptr;     // getImages from uint8: b / 255.0f for b = 0..255 (preproc.cu)
};

enum { MPN_CAT_CONV_TC = 0, MPN_CAT_CONV_DIRECT = 1, MPN_CAT_ROI = 2, MPN_CAT_NMS = 3, MPN_CAT_ELTWISE = 4, MPN_CAT_POOL = 5, MPN_NCAT = 6 };

// RAII: when ctx->profiling is on, brackets the launches issued in its scope with two events on the ctx stream.
struct MpnProfScope {
  mpn_ctx *ctx; int idx = -1;
  MpnProfScope(mpn_ctx *c, int cat) : ctx(c) {
    if (!c->profiling) return;
    auto get = [&]() { cudaEvent_t e; if (c->ev_pool.empty()) cudaEventCreate(&e); else { e = c->ev_pool.back(); c->ev_pool.pop_back(); } return e; };
    mpn_ctx::ProfRec r{cat, get(), get()};
    cudaEventRecord(r.a, c->stream);
    c->prof.push_back(r); idx = (int)c->prof.size() - 1;
  }
  ~MpnProfScope() { if (idx >= 0) cudaEventRecord(ctx->prof[idx].b, ctx->stream); }
};

#define MPN_OK 0
#define MPN_ERR_ARG (-1)
#define MPN_ERR_CUDA (-2)
#define MPN_ERR_STATE (-3)

inline int mpn_fail(mpn_ctx *ctx, int code, const std::string &msg) {
  if (ctx) ctx->err = msg;
  return code;
}

#define MPN_CUDA(ctx, expr)                                                         \
  do {                                                                              \
    cudaError_t e__ = (expr);                                                       \
    if (e__ != cudaSuccess) {                                                       \
      char b__[512];                                                                \
      snprintf(b__, sizeof b__, "CUDA error %s at %s:%d: %s", cudaGetErrorName(e__), \
               __FILE__, __LINE__, cudaGetErrorString(e__));                        \
      cudaGetLastError();                                                           \
      return mpn_fail((ctx), MPN_ERR_CUDA, b__);                                    \
    }                                                                               \
  } while (0)

#define MPN_CHECK_ARG(ctx, cond, msg)                                   \
  do {                                                                  \
    if (!(cond)) return mpn_fail((ctx), MPN_ERR_ARG, std::string(msg)); \
  } while (0)

#define MPN_TRY(expr)           \
  do {                          \
    int r__ = (expr);           \
    if (r__ != MPN_OK) return r__; \
  } while (0)

// count + check a kernel launch
#define MPN_LAUNCHED(ctx)                 \
  do {                                    \
    (ctx)->launches++;                    \
    MPN_CUDA((ctx), cudaGetLastError());  \
  } while (0)

// ---- programmatic dependent launch for the short kernels of the detect tail: the launch latency and prologue of kernel
// i+1 overlap kernel i. A kernel launched through mpn_launch_pdl MUST start with MPN_PDL_SYNC() (nothing global is read
// or written before the previous grid has completed and flushed); MPN_TC_PDL=0 turns the attribute off.
#define MPN_PDL_SYNC()                                                  \
  do {                                                                  \
    asm volatile("griddepcontrol.wait;" ::: "memory");                  \
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");     \
  } while (0)
inline bool mpn_pdl_enabled() {
  static const int on = [] { const char *e = getenv("MPN_TC_PDL"); return (e && e[0] == '0') ? 0 : 1; }();
  return on != 0;
}
template <typename... KArgs, typename... Args>
inline cudaError_t mpn_launch_pdl(mpn_ctx *ctx, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, Args &&...args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = ctx->stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = mpn_pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

// bits of the device flag word: an fp16 activation plane saturated / a ROI row named an image outside [1, N]
enum { MPN_FLAG_FP16_OVF = 1u, MPN_FLAG_BAD_BATCH = 2u };
int mpn_ovf_flag(mpn_ctx *ctx, unsigned **flag_dev);          // the ctx's device flag word (allocated on first use)
// enqueue the copy of the flag to its pinned host word on `stream` (no-op without a flag) / after that stream was
// synchronised: fail loudly if a flag bit was raised since the last test, and re-arm the flag
int mpn_ovf_copy_async(mpn_ctx *ctx, cudaStream_t stream);
int mpn_ovf_test(mpn_ctx *ctx);
int mpn_scratch(mpn_ctx *ctx, size_t bytes, void **out);    // slot 1
int mpn_scratch2(mpn_ctx *ctx, size_t bytes, void **out);   // slot 2
int mpn_scratch3(mpn_ctx *ctx, size_t bytes, void **out);   // slot 3

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---- split-bf16 representation ------------------------------------------------
// Every activation / weight that feeds the tensor cores is stored as two bf16
// planes: hi = bf16_rn(x), lo = bf16_rn(x - hi). hi + lo reproduces x to ~2^-17
// relative; the GEMMs issue hi*hi + lo*hi + hi*lo with fp32 accumulation in TMEM.
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16 &hi, __nv_bfloat16 &lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}
// two values at once: one packed conversion per plane (cvt.rn.bf16x2.f32), low half = first value
__device__ __forceinline__ void split_bf16x2(float x0, float x1, uint32_t &hi2, uint32_t &lo2) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);
  hi2 = *reinterpret_cast<const uint32_t *>(&h);
  const float r0 = x0 - __uint_as_float(hi2 << 16), r1 = x1 - __uint_as_float(hi2 & 0xffff0000u);
  const __nv_bfloat162 l = __floats2bfloat162_rn(r0, r1);
  lo2 = *reinterpret_cast<const uint32_t *>(&l);
}
// ---- fp16 split planes (DTensor::fmt == 1): hi = rn_f16(x), lo = rn_f16(x - hi): 22 significant bits for |x| >= 2^-3,
// an absolute 2^-24 below (fp16 subnormals), |x| <= 65504. Out-of-range (or NaN) inputs saturate and raise *ovf.
__device__ __forceinline__ void split_f16x2(float x0, float x1, uint32_t &hi2, uint32_t &lo2, unsigned *ovf) {
  const float c0 = fminf(fmaxf(x0, -65504.f), 65504.f), c1 = fminf(fmaxf(x1, -65504.f), 65504.f);
  if (ovf && (c0 != x0 || c1 != x1)) atomicOr(ovf, 1u);
  const __half2 h = __floats2half2_rn(c0, c1);
  hi2 = *reinterpret_cast<const uint32_t *>(&h);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(c0 - hf.x, c1 - hf.y);
  lo2 = *reinterpret_cast<const uint32_t *>(&l);
}
// one output pair in the tensor's plane format (fmt: 0 = bf16 hi/lo, 1 = fp16 hi/lo)
__device__ __forceinline__ void split_x2(int fmt, float x0, float x1, uint32_t &hi2, uint32_t &lo2, unsigned *ovf) {
  if (fmt) split_f16x2(x0, x1, hi2, lo2, ovf);
  else split_bf16x2(x0, x1, hi2, lo2);
}
__device__ __forceinline__ float join_planes(int fmt, uint16_t hi, uint16_t lo) {
  if (fmt) return __half2float(__ushort_as_half(hi)) + __half2float(__ushort_as_half(lo));
  return __uint_as_float((uint32_t)hi << 16) + __uint_as_float((uint32_t)lo << 16);
}
__device__ __forceinline__ float join_bf16(__nv_bfloat16 hi, __nv_bfloat16 lo) {
  return __bfloat162float(hi) + __bfloat162float(lo);
}
__device__ __forceinline__ float bf16_bits_to_float(uint32_t b16) { return __uint_as_float(b16 << 16); }
// unpack a uint32 holding two bf16 (low = element 0)
__device__ __forceinline__ float2 bf16x2_to_float2(uint32_t v) {
  return make_float2(__uint_as_float(v << 16), __uint_as_float(v & 0xffff0000u));
}
__device__ __forceinline__ uint32_t pack_bf16x2(__nv_bfloat16 a, __nv_bfloat16 b) {
  return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b) << 16);
}

// A device tensor in the library's internal layout: NHWC, either split-bf16 planes
// (hi, lo) or fp32, with a pixel stride `ld` (elements) so channel slices alias.
struct DTensor {
  __nv_bfloat16 *hi = nullptr, *lo = nullptr;   // 16-bit planes: bf16 (fmt 0) or fp16 (fmt 1) bit patterns
  int fmt = 0;
  float *f32 = nullptr;
  int64_t N = 0, H = 0, W = 0, C = 0, ld = 0;
  int64_t pixels() const { return N * H * W; }
};

// The images of a batched detect tail (mpn_model_detect_nms_batch*), passed by value to its kernels: image i owns proposal
// rows [off[i], off[i + 1]) and has its own im_scale and original size.
struct MpnBatch {
  int n;
  int off[MPN_MAX_BATCH + 1];
  float scale[MPN_MAX_BATCH], W0[MPN_MAX_BATCH], H0[MPN_MAX_BATCH];
};
__device__ __forceinline__ int mpn_batch_image(const MpnBatch &b, int64_t row) {   // the image owning proposal row `row`
  int i = 0;
  while (i + 1 < b.n && row >= b.off[i + 1]) ++i;
  return i;
}
