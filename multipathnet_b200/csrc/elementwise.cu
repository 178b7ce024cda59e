// elementwise.cu — the HBM-bound glue kernels of the detection path (sm_100a):
// region generation (Foveal/ContextRegion), BBoxNorm, bbox decode (+clamp), softmax
// (+ integral-head mean), per-class scored-box gather, max/avg pooling on split-bf16
// NHWC planes and layout converters. Each kernel cites the reference lines it restates.
#include "common.cuh"
#include <cuda_fp16.h>
#include <algorithm>
#include <float.h>

namespace {

// ---- nn.Foveal (modules/Foveal.lua:15-44): fp64 arithmetic, one rounding to fp32 ------
__global__ void foveal_kernel(const float *__restrict__ rois, int64_t R, float *__restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= R) return;
  const float *b = rois + i * 5;
  double id = b[0], x = b[1], y = b[2], x2 = b[3], y2 = b[4];
  double w = x2 - x, h = y2 - y;
  float *o = out + i * 20;
  o[0] = b[0]; o[1] = b[1]; o[2] = b[2]; o[3] = b[3]; o[4] = b[4];
  const double off[3] = {0.25, 0.5, 1.5}, mul[3] = {1.5, 2.0, 4.0};
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    double rx = __dsub_rn(x, __dmul_rn(w, off[k])), ry = __dsub_rn(y, __dmul_rn(h, off[k]));
    double rw = __dmul_rn(w, mul[k]), rh = __dmul_rn(h, mul[k]);
    float *q = o + 5 * (k + 1);
    q[0] = (float)id; q[1] = (float)rx; q[2] = (float)ry;
    q[3] = (float)__dadd_rn(rx, rw); q[4] = (float)__dadd_rn(ry, rh);
  }
}

// ---- nn.ContextRegion (modules/ContextRegion.lua:14-32): fp32 mm with [[a,0,b,0],...] -
__global__ void context_region_kernel(const float *__restrict__ rois, int64_t R, float a, float b,
                                      float *__restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= R) return;
  const float *r = rois + i * 5; float *o = out + i * 5;
  o[0] = r[0];
  o[1] = __fadd_rn(__fmul_rn(r[1], a), __fmul_rn(r[3], b));
  o[2] = __fadd_rn(__fmul_rn(r[2], a), __fmul_rn(r[4], b));
  o[3] = __fadd_rn(__fmul_rn(r[1], b), __fmul_rn(r[3], a));
  o[4] = __fadd_rn(__fmul_rn(r[2], b), __fmul_rn(r[4], a));
}

// ---- nn.BBoxNorm eval (modules/BBoxNorm.lua:27-28): x*std + mean over view(-1,4) -------
__global__ void bbox_norm_kernel(float *__restrict__ d, int64_t n4, float4 mean, float4 stdv) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  float4 v = reinterpret_cast<float4 *>(d)[i];
  v.x = __fadd_rn(__fmul_rn(v.x, stdv.x), mean.x);
  v.y = __fadd_rn(__fmul_rn(v.y, stdv.y), mean.y);
  v.z = __fadd_rn(__fmul_rn(v.z, stdv.z), mean.z);
  v.w = __fadd_rn(__fmul_rn(v.w, stdv.w), mean.w);
  reinterpret_cast<float4 *>(d)[i] = v;
}

// ---- utils.convertFrom per class block (utils.lua:226-246, ImageDetect.lua:183-185) ----
// optional clamp of Tester_FRCNN.lua:75-78 (x to [1,W0], y to [1,H0]).
// has_norm: apply nn.BBoxNorm (BBoxNorm.lua: y*std + mean, same op order as bbox_norm_kernel) to the raw deltas first
__device__ __forceinline__ void bbox_decode_body(int64_t idx, const float *__restrict__ deltas, const float *__restrict__ boxes,
                                                 int64_t R, int C, int do_clamp, float W0, float H0, float *__restrict__ out,
                                                 int has_norm, float4 mean, float4 stdv) {
  if (idx >= R * C) return;
  int64_t i = idx / C;
  float4 b = reinterpret_cast<const float4 *>(boxes)[i];
  float4 y = reinterpret_cast<const float4 *>(deltas)[idx];
  if (has_norm) {
    y.x = __fadd_rn(__fmul_rn(y.x, stdv.x), mean.x); y.y = __fadd_rn(__fmul_rn(y.y, stdv.y), mean.y);
    y.z = __fadd_rn(__fmul_rn(y.z, stdv.z), mean.z); y.w = __fadd_rn(__fmul_rn(y.w, stdv.w), mean.w);
  }
  float xc = __fmul_rn(__fadd_rn(b.x, b.z), 0.5f), yc = __fmul_rn(__fadd_rn(b.y, b.w), 0.5f);
  float w = __fsub_rn(b.z, b.x), h = __fsub_rn(b.w, b.y);
  float xtc = __fadd_rn(xc, __fmul_rn(y.x, w)), ytc = __fadd_rn(yc, __fmul_rn(y.y, h));
  float wt = __fmul_rn(expf(y.z), w), ht = __fmul_rn(expf(y.w), h);
  float hw = __fmul_rn(wt, 0.5f), hh = __fmul_rn(ht, 0.5f);
  float4 o = make_float4(__fsub_rn(xtc, hw), __fsub_rn(ytc, hh), __fadd_rn(xtc, hw), __fadd_rn(ytc, hh));
  if (do_clamp) {
    o.x = o.x < 1.f ? 1.f : (o.x > W0 ? W0 : o.x);
    o.z = o.z < 1.f ? 1.f : (o.z > W0 ? W0 : o.z);
    o.y = o.y < 1.f ? 1.f : (o.y > H0 ? H0 : o.y);
    o.w = o.w < 1.f ? 1.f : (o.w > H0 ? H0 : o.w);
  }
  reinterpret_cast<float4 *>(out)[idx] = o;
}
__global__ void bbox_decode_kernel(const float *__restrict__ deltas, const float *__restrict__ boxes,
                                   int64_t R, int C, int do_clamp, float W0, float H0,
                                   float *__restrict__ out) {
  bbox_decode_body((int64_t)blockIdx.x * blockDim.x + threadIdx.x, deltas, boxes, R, C, do_clamp, W0, H0, out, 0,
                   make_float4(0, 0, 0, 0), make_float4(1, 1, 1, 1));
}

// ---- nn.SoftMax over classes; with K>1 heads: mean over K of the K softmaxes ------------
// (ImageDetect.lua:189-191; integral eval branch model_utils.lua:296-313). One warp per ROI.
// logits laid out [K][R][C]. do_softmax=0 copies head 0 (model.noSoftMax with a single head).
__device__ __forceinline__ void softmax_mean_body(int64_t tid, const float *__restrict__ logits, int64_t R, int C, int K,
                                                  int do_softmax, float *__restrict__ out) {
  int64_t row = tid >> 5;
  int lane = (int)(tid & 31);
  if (row >= R) return;
  if (!do_softmax) {
    for (int c = lane; c < C; c += 32) out[row * C + c] = logits[row * C + c];
    return;
  }
  for (int c0 = 0; c0 < C; c0 += 32) {   // accumulate the mean chunk by chunk (C <= a few hundred)
    int c = c0 + lane;
    float acc = 0.f;
    for (int k = 0; k < K; ++k) {
      const float *x = logits + ((int64_t)k * R + row) * C;
      float m = -FLT_MAX;
      for (int cc = lane; cc < C; cc += 32) m = fmaxf(m, x[cc]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
      float s = 0.f;
      for (int cc = lane; cc < C; cc += 32) s += expf(x[cc] - m);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (c < C) acc += expf(x[c] - m) / s;
    }
    if (c < C) out[row * C + c] = (K > 1) ? acc / (float)K : acc;
  }
}
__global__ void softmax_mean_kernel(const float *__restrict__ logits, int64_t R, int C, int K,
                                    int do_softmax, float *__restrict__ out) {
  softmax_mean_body((int64_t)blockIdx.x * blockDim.x + threadIdx.x, logits, R, C, K, do_softmax, out);
}
// detect tail in ONE launch: blocks [0, nb_sm) = class_values (softmax / mean of softmaxes), the rest = BBoxNorm + decode (+clamp)
__global__ void __launch_bounds__(256)
detect_tail_kernel(const float *__restrict__ logits, int64_t R, int C, int K, int do_softmax, float *__restrict__ scores,
                   int nb_sm, const float *__restrict__ deltas, const float *__restrict__ boxes, int do_clamp, float W0,
                   float H0, float *__restrict__ bboxes, int has_norm, float4 mean, float4 stdv) {
  MPN_PDL_SYNC();
  if ((int)blockIdx.x < nb_sm) softmax_mean_body((int64_t)blockIdx.x * 256 + threadIdx.x, logits, R, C, K, do_softmax, scores);
  else bbox_decode_body((int64_t)(blockIdx.x - nb_sm) * 256 + threadIdx.x, deltas, boxes, R, C, do_clamp, W0, H0, bboxes, has_norm, mean, stdv);
}

// batched detect tail: the same blocks, every decoded row clamped to its own image's W0 x H0 (Tester_FRCNN.lua:75-78)
__global__ void __launch_bounds__(256)
detect_tail_batch_kernel(const float *__restrict__ logits, int64_t R, int C, int K, int do_softmax, float *__restrict__ scores,
                         int nb_sm, const float *__restrict__ deltas, const float *__restrict__ boxes, const MpnBatch b,
                         float *__restrict__ bboxes, int has_norm, float4 mean, float4 stdv) {
  MPN_PDL_SYNC();
  if ((int)blockIdx.x < nb_sm) { softmax_mean_body((int64_t)blockIdx.x * 256 + threadIdx.x, logits, R, C, K, do_softmax, scores); return; }
  const int64_t idx = (int64_t)(blockIdx.x - nb_sm) * 256 + threadIdx.x;
  const int img = mpn_batch_image(b, idx / C);
  bbox_decode_body(idx, deltas, boxes, R, C, 1, b.W0[img], b.H0[img], bboxes, has_norm, mean, stdv);
}

// ---- Tester_FRCNN.lua:106-116: per foreground class j gather rows with score > thresh ----
// into seg j-1: sb[seg][k] = [bbox(:,4j..4j+3), score(:,j)], order preserved (stable), plus
// src_idx[seg][k] = original ROI row and counts[seg]. One block per class.
// body for one (image, class) segment: rows [0, R) of scores / bboxes, class j, outputs at sb / src_idx (capacity >= R)
__device__ __forceinline__ void gather_scored_body(const float *__restrict__ scores, const float *__restrict__ bboxes, int R, int C,
                                                   int j, float thresh, float *__restrict__ sb, int32_t *__restrict__ src_idx,
                                                   int32_t *__restrict__ count) {
  __shared__ int s_wtot[8];
  __shared__ int s_total;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int base_out = 0;
  for (int r0 = 0; r0 < R; r0 += 256) {
    int r = r0 + threadIdx.x;
    float s = 0.f; int flag = 0;
    if (r < R) { s = scores[(size_t)r * C + j]; flag = (s > thresh) ? 1 : 0; }
    unsigned ball = __ballot_sync(0xffffffffu, flag);
    int pre = __popc(ball & ((1u << lane) - 1u));
    if (lane == 0) s_wtot[wid] = __popc(ball);
    __syncthreads();
    if (threadIdx.x == 0) {
      int acc = 0;
      for (int w = 0; w < 8; ++w) { int t = s_wtot[w]; s_wtot[w] = acc; acc += t; }
      s_total = acc;
    }
    __syncthreads();
    if (flag) {
      int k = base_out + s_wtot[wid] + pre;
      float4 b = reinterpret_cast<const float4 *>(bboxes)[(size_t)r * C + j];
      float *o = sb + (size_t)k * 5;
      o[0] = b.x; o[1] = b.y; o[2] = b.z; o[3] = b.w; o[4] = s;
      src_idx[k] = r;
    }
    base_out += s_total;
    __syncthreads();
  }
  if (threadIdx.x == 0) *count = base_out;
}
__global__ void __launch_bounds__(256)
gather_scored_kernel(const float *__restrict__ scores, const float *__restrict__ bboxes, int R, int C,
                     float thresh, float *__restrict__ sb, int32_t *__restrict__ src_idx,
                     int32_t *__restrict__ counts) {
  MPN_PDL_SYNC();
  const int seg = blockIdx.x;
  gather_scored_body(scores, bboxes, R, C, seg + 1, thresh, sb + (size_t)seg * R * 5, src_idx + (size_t)seg * R, counts + seg);
}
// batched form: grid (C - 1, N); segment (image i, class j) = i * (C - 1) + j - 1 at capacity cap, row indices local to image i
__global__ void __launch_bounds__(256)
gather_scored_batch_kernel(const float *__restrict__ scores, const float *__restrict__ bboxes, int C, float thresh, const MpnBatch b,
                           int cap, float *__restrict__ sb, int32_t *__restrict__ src_idx, int32_t *__restrict__ counts) {
  MPN_PDL_SYNC();
  const int img = blockIdx.y, r0 = b.off[img];
  const size_t seg = (size_t)img * (C - 1) + blockIdx.x;
  gather_scored_body(scores + (size_t)r0 * C, bboxes + (size_t)r0 * 4 * C, b.off[img + 1] - r0, C, blockIdx.x + 1, thresh,
                     sb + seg * cap * 5, src_idx + seg * cap, counts + seg);
}

// ---- max-pool k x k / stride / pad on split-bf16 NHWC planes, 8 channels per thread ------
// (nn.SpatialMaxPooling; Caffe-converted VGG uses ceil mode: SURVEY 8a5). Windows are
// clipped to the input (padding never wins a max).
__global__ void maxpool_split_kernel(const __nv_bfloat16 *__restrict__ ih, const __nv_bfloat16 *__restrict__ il,
                                     int N, int H, int W, int C, int64_t ld_in, int k, int s, int p,
                                     int Ho, int Wo, __nv_bfloat16 *__restrict__ oh,
                                     __nv_bfloat16 *__restrict__ ol, int64_t ld_out) {
  const int cg = C >> 3;
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = (int64_t)N * Ho * Wo * cg;
  if (idx >= total) return;
  int c8 = (int)(idx % cg); int64_t pix = idx / cg;
  int wo = (int)(pix % Wo); int ho = (int)((pix / Wo) % Ho); int n = (int)(pix / ((int64_t)Wo * Ho));
  int h0 = ho * s - p, w0 = wo * s - p;
  int h1 = min(h0 + k, H), w1 = min(w0 + k, W);
  h0 = max(h0, 0); w0 = max(w0, 0);
  float m[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) m[e] = -FLT_MAX;
  for (int h = h0; h < h1; ++h)
    for (int w = w0; w < w1; ++w) {
      int64_t off = (((int64_t)n * H + h) * W + w) * ld_in + c8 * 8;
      uint4 vh = *reinterpret_cast<const uint4 *>(ih + off);
      uint4 vl = *reinterpret_cast<const uint4 *>(il + off);
      const uint32_t hh[4] = {vh.x, vh.y, vh.z, vh.w}, ll[4] = {vl.x, vl.y, vl.z, vl.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float2 a = bf16x2_to_float2(hh[q]), b = bf16x2_to_float2(ll[q]);
        m[2 * q] = fmaxf(m[2 * q], a.x + b.x);
        m[2 * q + 1] = fmaxf(m[2 * q + 1], a.y + b.y);
      }
    }
  uint32_t ph[4], pl[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    __nv_bfloat16 h0b, l0b, h1b, l1b;
    split_bf16(m[2 * q], h0b, l0b); split_bf16(m[2 * q + 1], h1b, l1b);
    ph[q] = pack_bf16x2(h0b, h1b); pl[q] = pack_bf16x2(l0b, l1b);
  }
  int64_t o = pix * ld_out + c8 * 8;
  *reinterpret_cast<uint4 *>(oh + o) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
  *reinterpret_cast<uint4 *>(ol + o) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
}

// ---- global average pool over H x W (ResNet avgpool 7, resnet.lua:39) ---------------------
__global__ void avgpool_split_kernel(const __nv_bfloat16 *__restrict__ ih, const __nv_bfloat16 *__restrict__ il,
                                     int N, int HW, int C, int64_t ld_in, __nv_bfloat16 *__restrict__ oh,
                                     __nv_bfloat16 *__restrict__ ol, int64_t ld_out) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)N * C) return;
  int c = (int)(idx % C); int64_t n = idx / C;
  float s = 0.f;
  for (int p = 0; p < HW; ++p) {
    int64_t off = (n * HW + p) * ld_in + c;
    s += join_bf16(ih[off], il[off]);
  }
  s = s / (float)HW;
  __nv_bfloat16 h, l; split_bf16(s, h, l);
  oh[n * ld_out + c] = h; ol[n * ld_out + c] = l;
}

// ---- layout converters ---------------------------------------------------------------------
// fp32 [rows][cols] (row stride ld_in) -> split planes [rows][ld_out]
__global__ void split_rows_kernel(const float *__restrict__ in, int64_t rows, int64_t cols, int64_t ld_in,
                                  __nv_bfloat16 *__restrict__ oh, __nv_bfloat16 *__restrict__ ol, int64_t ld_out) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * cols) return;
  int64_t r = idx / cols, c = idx % cols;
  __nv_bfloat16 h, l; split_bf16(in[r * ld_in + c], h, l);
  oh[r * ld_out + c] = h; ol[r * ld_out + c] = l;
}
// split planes [rows][ld_in] (fmt 0 = bf16, 1 = fp16) -> fp32 [rows][cols] (hi + lo: exact in fp32)
__global__ void join_rows_kernel(const __nv_bfloat16 *__restrict__ ih, const __nv_bfloat16 *__restrict__ il, int64_t rows,
                                 int64_t cols, int64_t ld_in, int fmt, float *__restrict__ out) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * cols) return;
  int64_t r = idx / cols, c = idx % cols;
  out[idx] = join_planes(fmt, __bfloat16_as_ushort(ih[r * ld_in + c]), __bfloat16_as_ushort(il[r * ld_in + c]));
}
// fp32 [rows][cols] -> fp16 split planes (tests of the "w16" kernels)
__global__ void split_rows_f16_kernel(const float *__restrict__ in, int64_t rows, int64_t cols, int64_t ld_in,
                                      __nv_bfloat16 *__restrict__ oh, __nv_bfloat16 *__restrict__ ol, int64_t ld_out, unsigned *ovf) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * cols) return;
  int64_t r = idx / cols, c = idx % cols;
  uint32_t h2, l2;
  split_f16x2(in[r * ld_in + c], 0.f, h2, l2, ovf);
  oh[r * ld_out + c] = __ushort_as_bfloat16((unsigned short)(h2 & 0xffffu)); ol[r * ld_out + c] = __ushort_as_bfloat16((unsigned short)(l2 & 0xffffu));
}
// NCHW fp32 -> NHWC split planes
__global__ void nchw_to_nhwc_split_kernel(const float *__restrict__ in, int N, int C, int H, int W,
                                          __nv_bfloat16 *__restrict__ oh, __nv_bfloat16 *__restrict__ ol, int64_t ld) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = (int64_t)N * C * H * W;
  if (idx >= total) return;
  int c = (int)(idx % C); int64_t pix = idx / C;
  int w = (int)(pix % W); int h = (int)((pix / W) % H); int n = (int)(pix / ((int64_t)W * H));
  float v = in[(((int64_t)n * C + c) * H + h) * W + w];
  __nv_bfloat16 hh, ll; split_bf16(v, hh, ll);
  oh[pix * ld + c] = hh; ol[pix * ld + c] = ll;
}
// NHWC split planes -> NCHW fp32
__global__ void nhwc_split_to_nchw_kernel(const __nv_bfloat16 *__restrict__ ih, const __nv_bfloat16 *__restrict__ il,
                                          int N, int C, int H, int W, int64_t ld, float *__restrict__ out) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = (int64_t)N * C * H * W;
  if (idx >= total) return;
  int w = (int)(idx % W); int h = (int)((idx / W) % H); int c = (int)((idx / ((int64_t)W * H)) % C);
  int n = (int)(idx / ((int64_t)W * H * C));
  int64_t pix = ((int64_t)n * H + h) * W + w;
  out[idx] = join_bf16(ih[pix * ld + c], il[pix * ld + c]);
}

// ---- ImageDetect.lua:66-70 project_im_rois: rois = [1, (box-1)*im_scale + 1] -----------------
__global__ void project_rois_kernel(const float *__restrict__ boxes, int64_t R, float im_scale,
                                    float *__restrict__ rois) {
  MPN_PDL_SYNC();
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= R) return;
  float4 b = reinterpret_cast<const float4 *>(boxes)[i];
  float *o = rois + i * 5;
  o[0] = 1.0f;
  o[1] = __fadd_rn(__fmul_rn(__fsub_rn(b.x, 1.0f), im_scale), 1.0f);
  o[2] = __fadd_rn(__fmul_rn(__fsub_rn(b.y, 1.0f), im_scale), 1.0f);
  o[3] = __fadd_rn(__fmul_rn(__fsub_rn(b.z, 1.0f), im_scale), 1.0f);
  o[4] = __fadd_rn(__fmul_rn(__fsub_rn(b.w, 1.0f), im_scale), 1.0f);
}

// batched form: row i belongs to image b(i), projected with that image's im_scale, batch index b(i) + 1
__global__ void project_rois_batch_kernel(const float *__restrict__ boxes, int64_t R, const MpnBatch bt, float *__restrict__ rois) {
  MPN_PDL_SYNC();
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= R) return;
  const int img = mpn_batch_image(bt, i);
  const float im_scale = bt.scale[img];
  float4 b = reinterpret_cast<const float4 *>(boxes)[i];
  float *o = rois + i * 5;
  o[0] = (float)(img + 1);
  o[1] = __fadd_rn(__fmul_rn(__fsub_rn(b.x, 1.0f), im_scale), 1.0f);
  o[2] = __fadd_rn(__fmul_rn(__fsub_rn(b.y, 1.0f), im_scale), 1.0f);
  o[3] = __fadd_rn(__fmul_rn(__fsub_rn(b.z, 1.0f), im_scale), 1.0f);
  o[4] = __fadd_rn(__fmul_rn(__fsub_rn(b.w, 1.0f), im_scale), 1.0f);
}

// ---- weight re-layout: Torch conv weight [Cout][Cin][kh][kw] fp32 -> [Cout][kh][kw][Cin] split bf16
__global__ void weight_permute_split_kernel(const float *__restrict__ w, int64_t Cout, int Cin, int kh, int kw,
                                            __nv_bfloat16 *__restrict__ oh, __nv_bfloat16 *__restrict__ ol) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t K = (int64_t)Cin * kh * kw;
  if (idx >= Cout * K) return;
  int64_t co = idx / K; int64_t k = idx % K;            // output order (r, q, ci)
  int ci = (int)(k % Cin); int q = (int)((k / Cin) % kw); int r = (int)(k / ((int64_t)Cin * kw));
  float v = w[((co * Cin + ci) * kh + r) * kw + q];
  __nv_bfloat16 h, l; split_bf16(v, h, l);
  oh[idx] = h; ol[idx] = l;
}

// max |w| of an fp32 array (bit pattern of a non-negative float orders like an unsigned integer); *out must start at 0
__global__ void absmax_kernel(const float *__restrict__ w, int64_t n, unsigned *__restrict__ out) {
  float m = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) m = fmaxf(m, fabsf(w[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(out, __float_as_uint(m));
}
// Torch conv weight [Cout][Cin][kh][kw] fp32 -> [Cout][kh][kw][Cin] ONE fp16 plane of w * scale (scale = a power of two)
__global__ void weight_permute_half_kernel(const float *__restrict__ w, int64_t Cout, int Cin, int kh, int kw, float scale,
                                           __half *__restrict__ o) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t K = (int64_t)Cin * kh * kw;
  if (idx >= Cout * K) return;
  int64_t co = idx / K; int64_t k = idx % K;            // output order (r, q, ci)
  int ci = (int)(k % Cin); int q = (int)((k / Cin) % kw); int r = (int)(k / ((int64_t)Cin * kw));
  o[idx] = __float2half_rn(w[((co * Cin + ci) * kh + r) * kw + q] * scale);
}

}  // namespace

static inline unsigned nblk(int64_t n, int t) { return (unsigned)((n + t - 1) / t); }

int mpn_foveal_launch(mpn_ctx *ctx, const float *rois_dev, int64_t R, float *out_dev) {
  if (R <= 0) return MPN_OK;
  foveal_kernel<<<nblk(R, 128), 128, 0, ctx->stream>>>(rois_dev, R, out_dev);
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
int mpn_context_region_launch(mpn_ctx *ctx, const float *rois_dev, int64_t R, float scale, float *out_dev) {
  if (R <= 0) return MPN_OK;
  float a = (float)((1.0 + (double)scale) / 2.0), b = (float)((1.0 - (double)scale) / 2.0);
  context_region_kernel<<<nblk(R, 128), 128, 0, ctx->stream>>>(rois_dev, R, a, b, out_dev);
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
int mpn_bbox_norm_launch(mpn_ctx *ctx, float *d_dev, int64_t R, int64_t C4, const float *mean4, const float *std4) {
  MpnProfScope prof_scope__(ctx, MPN_CAT_ELTWISE);
  int64_t n4 = R * C4 / 4;
  if (n4 <= 0) return MPN_OK;
  bbox_norm_kernel<<<nblk(n4, 256), 256, 0, ctx->stream>>>(
      d_dev, n4, make_float4(mean4[0], mean4[1], mean4[2], mean4[3]), make_float4(std4[0], std4[1], std4[2], std4[3]));
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
int mpn_bbox_decode_launch(mpn_ctx *ctx, const float *deltas_dev, const float *boxes_dev, int64_t R, int C,
                           int do_clamp, float W0, float H0, float *out_dev) {
  MpnProfScope prof_scope__(ctx, MPN_CAT_ELTWISE);
  if (R * C <= 0) return MPN_OK;
  bbox_decode_kernel<<<nblk(R * C, 256), 256, 0, ctx->stream>>>(deltas_dev, boxes_dev, R, C, do_clamp, W0, H0, out_dev);
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
int mpn_detect_tail_launch(mpn_ctx *ctx, const float *logits_dev, int64_t R, int C, int K, int do_softmax, float *scores_dev,
                           const float *deltas_dev, const float *boxes_dev, int do_clamp, float W0, float H0,
                           float *bboxes_dev, int has_norm, const float *mean4, const float *std4) {
  MpnProfScope prof_scope__(ctx, MPN_CAT_ELTWISE);
  if (R <= 0) return MPN_OK;
  const int nb_sm = (int)nblk(R * 32, 256), nb_dec = (int)nblk(R * C, 256);
  MPN_CUDA(ctx, mpn_launch_pdl(ctx, detect_tail_kernel, dim3(nb_sm + nb_dec), dim3(256), 0,
      logits_dev, R, C, K, do_softmax, scores_dev, nb_sm, deltas_dev, boxes_dev, do_clamp, W0, H0, bboxes_dev, has_norm,
      make_float4(mean4[0], mean4[1], mean4[2], mean4[3]), make_float4(std4[0], std4[1], std4[2], std4[3])));
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
int mpn_softmax_mean_launch(mpn_ctx *ctx, const float *logits_dev, int64_t R, int C, int K, int do_softmax,
                            float *out_dev) {
  MpnProfScope prof_scope__(ctx, MPN_CAT_ELTWISE);
  if (R <= 0) return MPN_OK;
  softmax_mean_kernel<<<nblk(R * 32, 256), 256, 0, ctx->stream>>>(logits_dev, R, C, K, do_softmax, out_dev);
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
int mpn_gather_scored_launch(mpn_ctx *ctx, const float *scores_dev, const float *bboxes_dev, int R, int C,
                             float thresh, float *sb_dev, int32_t *src_idx_dev, int32_t *counts_dev) {
  MpnProfScope prof_scope__(ctx, MPN_CAT_ELTWISE);
  if (C <= 1 || R <= 0) return MPN_OK;
  MPN_CUDA(ctx, mpn_launch_pdl(ctx, gather_scored_kernel, dim3(C - 1), dim3(256), 0, scores_dev, bboxes_dev, R, C, thresh, sb_dev, src_idx_dev, counts_dev));
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
// per-class gather for the foreground classes [c_begin, c_begin + nseg) only (1-based class index): segment s = class
// c_begin + s, capacity R each (class-sharded post-processing: BASELINE configs[4])
int mpn_gather_scored_range_launch(mpn_ctx *ctx, const float *scores_dev, const float *bboxes_dev, int R, int C, int c_begin, int nseg,
                                   float thresh, float *sb_dev, int32_t *src_idx_dev, int32_t *counts_dev) {
  MpnProfScope prof_scope__(ctx, MPN_CAT_ELTWISE);
  if (nseg <= 0 || R <= 0) return MPN_OK;
  // the kernel addresses class j = seg + 1 of row r as scores[r*C + j] / float4 bboxes[r*C + j]: shift both bases
  MPN_CUDA(ctx, mpn_launch_pdl(ctx, gather_scored_kernel, dim3(nseg), dim3(256), 0, scores_dev + (c_begin - 1), bboxes_dev + 4 * (size_t)(c_begin - 1),
                               R, C, thresh, sb_dev, src_idx_dev, counts_dev));
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
int mpn_bbox_norm_decode_launch(mpn_ctx *ctx, const float *deltas_dev, const float *boxes_dev, int64_t R, int C, int do_clamp, float W0,
                                float H0, float *out_dev, const float *mean4, const float *std4) {
  MpnProfScope prof_scope__(ctx, MPN_CAT_ELTWISE);
  if (R <= 0) return MPN_OK;
  const int has = (mean4 && std4) ? 1 : 0;
  MPN_CUDA(ctx, mpn_launch_pdl(ctx, detect_tail_kernel, dim3(nblk(R * C, 256)), dim3(256), 0, (const float *)nullptr, R, C, 1, 0, (float *)nullptr, 0,
      deltas_dev, boxes_dev, do_clamp, W0, H0, out_dev, has,
      has ? make_float4(mean4[0], mean4[1], mean4[2], mean4[3]) : make_float4(0, 0, 0, 0),
      has ? make_float4(std4[0], std4[1], std4[2], std4[3]) : make_float4(1, 1, 1, 1)));
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
int mpn_maxpool_launch(mpn_ctx *ctx, const DTensor &in, int k, int s, int p, DTensor &out) {
  MpnProfScope prof_scope__(ctx, MPN_CAT_POOL);
  int64_t total = out.N * out.H * out.W * (out.C / 8);
  if (total <= 0) return MPN_OK;
  maxpool_split_kernel<<<nblk(total, 256), 256, 0, ctx->stream>>>(in.hi, in.lo, (int)in.N, (int)in.H, (int)in.W, (int)in.C,
                                                               in.ld, k, s, p, (int)out.H, (int)out.W, out.hi, out.lo, out.ld);
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
int mpn_avgpool_launch(mpn_ctx *ctx, const DTensor &in, DTensor &out) {
  MpnProfScope prof_scope__(ctx, MPN_CAT_ELTWISE);
  int64_t total = in.N * in.C;
  if (total <= 0) return MPN_OK;
  avgpool_split_kernel<<<nblk(total, 256), 256, 0, ctx->stream>>>(in.hi, in.lo, (int)in.N, (int)(in.H * in.W), (int)in.C,
                                                               in.ld, out.hi, out.lo, out.ld);
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
int mpn_split_rows_launch(mpn_ctx *ctx, const float *in_dev, int64_t rows, int64_t cols, int64_t ld_in,
                          __nv_bfloat16 *oh, __nv_bfloat16 *ol, int64_t ld_out) {
  if (rows * cols <= 0) return MPN_OK;
  split_rows_kernel<<<nblk(rows * cols, 256), 256, 0, ctx->stream>>>(in_dev, rows, cols, ld_in, oh, ol, ld_out);
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
// max |w| (device array) -> host; synchronises the ctx stream (model-planning time only)
int mpn_absmax(mpn_ctx *ctx, const float *w_dev, int64_t n, float *out_host) {
  if (!ctx->small_dev) MPN_CUDA(ctx, cudaMalloc(&ctx->small_dev, 256));
  unsigned *d = (unsigned *)ctx->small_dev;
  MPN_CUDA(ctx, cudaMemsetAsync(d, 0, sizeof(unsigned), ctx->stream));
  if (n > 0) { absmax_kernel<<<(unsigned)std::min<int64_t>((n + 255) / 256, 1184), 256, 0, ctx->stream>>>(w_dev, n, d); MPN_LAUNCHED(ctx); }
  unsigned bits = 0;
  MPN_CUDA(ctx, cudaMemcpyAsync(&bits, d, sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  memcpy(out_host, &bits, sizeof(float));
  return MPN_OK;
}
int mpn_weight_permute_half_launch(mpn_ctx *ctx, const float *w_dev, int64_t Cout, int Cin, int kh, int kw, float scale, void *out) {
  int64_t total = Cout * Cin * kh * kw;
  if (total <= 0) return MPN_OK;
  weight_permute_half_kernel<<<nblk(total, 256), 256, 0, ctx->stream>>>(w_dev, Cout, Cin, kh, kw, scale, (__half *)out);
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
int mpn_split_rows_f16_launch(mpn_ctx *ctx, const float *in_dev, int64_t rows, int64_t cols, int64_t ld_in, __nv_bfloat16 *oh,
                              __nv_bfloat16 *ol, int64_t ld_out) {
  if (rows * cols <= 0) return MPN_OK;
  unsigned *ovf = nullptr;
  MPN_TRY(mpn_ovf_flag(ctx, &ovf));
  split_rows_f16_kernel<<<nblk(rows * cols, 256), 256, 0, ctx->stream>>>(in_dev, rows, cols, ld_in, oh, ol, ld_out, ovf);
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
int mpn_join_rows_launch(mpn_ctx *ctx, const __nv_bfloat16 *ih, const __nv_bfloat16 *il, int64_t rows, int64_t cols, int64_t ld_in,
                         int fmt, float *out_dev) {
  if (rows * cols <= 0) return MPN_OK;
  join_rows_kernel<<<nblk(rows * cols, 256), 256, 0, ctx->stream>>>(ih, il, rows, cols, ld_in, fmt, out_dev);
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
int mpn_nchw_to_nhwc_split_launch(mpn_ctx *ctx, const float *in_dev, int N, int C, int H, int W, DTensor &out) {
  int64_t total = (int64_t)N * C * H * W;
  if (total <= 0) return MPN_OK;
  nchw_to_nhwc_split_kernel<<<nblk(total, 256), 256, 0, ctx->stream>>>(in_dev, N, C, H, W, out.hi, out.lo, out.ld);
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
int mpn_nhwc_split_to_nchw_launch(mpn_ctx *ctx, const DTensor &in, float *out_dev) {
  int64_t total = in.N * in.C * in.H * in.W;
  if (total <= 0) return MPN_OK;
  nhwc_split_to_nchw_kernel<<<nblk(total, 256), 256, 0, ctx->stream>>>(in.hi, in.lo, (int)in.N, (int)in.C, (int)in.H,
                                                                    (int)in.W, in.ld, out_dev);
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}

int mpn_project_rois_launch(mpn_ctx *ctx, const float *boxes_dev, int64_t R, float im_scale, float *rois_dev) {
  MpnProfScope prof_scope__(ctx, MPN_CAT_ELTWISE);
  if (R <= 0) return MPN_OK;
  MPN_CUDA(ctx, mpn_launch_pdl(ctx, project_rois_kernel, dim3(nblk(R, 128)), dim3(128), 0, boxes_dev, R, im_scale, rois_dev));
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
int mpn_project_rois_batch_launch(mpn_ctx *ctx, const float *boxes_dev, int64_t R, const MpnBatch &b, float *rois_dev) {
  MpnProfScope prof_scope__(ctx, MPN_CAT_ELTWISE);
  if (R <= 0) return MPN_OK;
  MPN_CUDA(ctx, mpn_launch_pdl(ctx, project_rois_batch_kernel, dim3(nblk(R, 128)), dim3(128), 0, boxes_dev, R, b, rois_dev));
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
int mpn_detect_tail_batch_launch(mpn_ctx *ctx, const float *logits_dev, int64_t R, int C, int K, int do_softmax, float *scores_dev,
                                 const float *deltas_dev, const float *boxes_dev, const MpnBatch &b, float *bboxes_dev, int has_norm,
                                 const float *mean4, const float *std4) {
  MpnProfScope prof_scope__(ctx, MPN_CAT_ELTWISE);
  if (R <= 0) return MPN_OK;
  const int nb_sm = (int)nblk(R * 32, 256), nb_dec = (int)nblk(R * C, 256);
  MPN_CUDA(ctx, mpn_launch_pdl(ctx, detect_tail_batch_kernel, dim3(nb_sm + nb_dec), dim3(256), 0,
      logits_dev, R, C, K, do_softmax, scores_dev, nb_sm, deltas_dev, boxes_dev, b, bboxes_dev, has_norm,
      make_float4(mean4[0], mean4[1], mean4[2], mean4[3]), make_float4(std4[0], std4[1], std4[2], std4[3])));
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
int mpn_gather_scored_batch_launch(mpn_ctx *ctx, const float *scores_dev, const float *bboxes_dev, int C, float thresh, const MpnBatch &b,
                                   int cap, float *sb_dev, int32_t *src_idx_dev, int32_t *counts_dev) {
  MpnProfScope prof_scope__(ctx, MPN_CAT_ELTWISE);
  if (C <= 1 || b.n <= 0) return MPN_OK;
  MPN_CUDA(ctx, mpn_launch_pdl(ctx, gather_scored_batch_kernel, dim3(C - 1, b.n), dim3(256), 0, scores_dev, bboxes_dev, C, thresh, b, cap,
                               sb_dev, src_idx_dev, counts_dev));
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
int mpn_weight_permute_split_launch(mpn_ctx *ctx, const float *w_dev, int64_t Cout, int Cin, int kh, int kw,
                                    __nv_bfloat16 *oh, __nv_bfloat16 *ol) {
  int64_t total = Cout * Cin * kh * kw;
  if (total <= 0) return MPN_OK;
  weight_permute_split_kernel<<<nblk(total, 256), 256, 0, ctx->stream>>>(w_dev, Cout, Cin, kh, kw, oh, ol);
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}
