// roi.cuh — job descriptors of the fused Foveal + ROI-pooling kernel (roi.cu), shared with model.cu
#pragma once
#include "common.cuh"
constexpr int ROI_MAX_LEVELS = 6;   // level 0 = the feature map, level k = max over 2^k x 2^k blocks at every position
struct RoiJob {
  // max pyramid of the feature map as fp32 NHWC (pixel stride C): level 0 = the joined map itself, level k = max over the
  // 2^k x 2^k block starting at every position. fp32 costs the same bytes as the hi+lo planes and lets the pooling
  // kernel take maxima straight from the loads (it is instruction-issue bound, not bandwidth bound).
  const float *lv[ROI_MAX_LEVELS];
  int nlev;                        // number of valid levels incl. level 0
  int H, W, C;
  int nimg;                        // images in the pyramid (image stride H * W * C); a ROI naming another raises MPN_FLAG_BAD_BATCH
  unsigned *flag;                  // the ctx's device flag word
  float scale;                     // spatial scale
  int region;                      // 0: ROI, 1..3: foveal x1.5, x2, x4
  __nv_bfloat16 *out_hi, *out_lo;  // R x bins x out_ld
  long long out_ld; int out_ch_off;
  int tower;                       // host bookkeeping: index of the tower this job pools for
  int out_fmt; unsigned *ovf;      // plane format of the pooled tensor (0 = bf16 split, 1 = fp16 split: feeds a "w16" Linear)
  int normalize;
};
constexpr int MAX_ROI_JOBS = 16;
struct RoiJobs { RoiJob j[MAX_ROI_JOBS]; int n; };
int mpn_roi_pool_fused_launch(mpn_ctx *ctx, const RoiJobs &jobs, const float *rois_dev, int64_t R, int PW, int PH,
                              int variant);
// level 0: join the split planes (pixel stride ld_in) into fp32 [pix][C]
int mpn_pyr_level0_launch(mpn_ctx *ctx, const __nv_bfloat16 *ph, const __nv_bfloat16 *pl, int N, int H, int W, int C, long long ld_in,
                          float *out);
// level k (block 2^k) from level k-1: out[y][x] = max of the four 2^(k-1) blocks at (y,x),(y,x+s),(y+s,x),(y+s,x+s)
int mpn_maxpyr_launch(mpn_ctx *ctx, const float *prev, int N, int H, int W, int C, int s, float *out);
// every level (0..nlev-1) of a small map in one launch; *too_big = 1 (nothing launched) when the plane does not fit in smem
int mpn_maxpyr_all_launch(mpn_ctx *ctx, const __nv_bfloat16 *ph, const __nv_bfloat16 *pl, int N, int H, int W, int C,
                          long long ld_in, int nlev, float *const *out, int *too_big);
int mpn_roi_pool_nchw_launch(mpn_ctx *ctx, const float *fmap_dev, int64_t N, int64_t C, int64_t H, int64_t W,
                             const float *rois_dev, int64_t R, int PW, int PH, float scale, int variant,
                             float *out_dev, int32_t *argmax_dev);
