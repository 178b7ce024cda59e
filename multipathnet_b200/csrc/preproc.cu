// getImages on the device (SURVEY 8f-1): ImageTransformer + image.scale fused into one HBM-bound kernel, for one image or
// for N images into one zero-padded N x 3 x H x W canvas (ImageDetect.lua:44-50).
// Reference: ImageDetect.lua:22-52, modules/ImageTransformer.lua:19-33; the arithmetic lives in image_scale.cuh
// (shared with the CPU suite). One thread per canvas element of the 3 x H x W plane of image n, x fastest so the store is
// coalesced; the 4 .. (f+2)^2 source reads of neighbouring threads overlap and are served by L1 / L2 (the raw images are
// a few MB, far below the 126 MB L2). Algorithmic bytes: sum_i 3*H0_i*W0_i (uint8) or *4 (fp32) read + N*3*H*W*4 written
// (the padding zeros included: the kernel writes every element, so no memset precedes it). A single image is N = 1 with
// the canvas equal to the image.
#include "common.cuh"
#include "image_scale.cuh"

static_assert((int)mpn_img::kMaxBatchImages == (int)MPN_MAX_BATCH, "image_scale.cuh's batch capacity is MPN_MAX_BATCH");

// per-image parameters (source offset, sizes, the two axis steps sx / sy divided once on the host: same IEEE division =>
// same bits as the per-pixel division of the first version, which spent most of its ~300 instructions per pixel in three
// fdivs: 20.8 us for 480x640 -> 600x800) live in the __grid_constant__ struct, read in place from parameter space.
// Min 4 blocks / SM: without it the per-image fields take the kernel from 64 to 74 registers (3 blocks / SM); with it, 60
// and no spills.
__global__ void __launch_bounds__(256, 4) get_images_kernel(const __grid_constant__ mpn_img::ImageBatch B, float *__restrict__ out) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  const int n = blockIdx.z / 3, c = blockIdx.z - 3 * n;
  if (x >= B.W) return;
  out[(((int64_t)n * 3 + c) * B.H + y) * B.W + x] = mpn_img::batch_pixel(B, n, c, y, x);
}

// ImageDetect.lua:31-39: im_scale = scale / min(H0, W0), capped so that round(im_scale * max(H0, W0)) <= max_size;
// image.scale receives H0*im_scale, W0*im_scale as Lua numbers and allocates the result with them truncated to long.
int mpn_get_images_size_impl(int32_t H0, int32_t W0, double scale, double max_size, int32_t *h, int32_t *w, double *im_scale) {
  if (H0 <= 0 || W0 <= 0 || !(scale > 0) || !(max_size > 0)) return MPN_ERR_ARG;
  const double smin = H0 < W0 ? H0 : W0, smax = H0 < W0 ? W0 : H0;
  double s = scale / smin;
  if (floor(s * smax + 0.5) > max_size) s = max_size / smax;    // torch.round: half away from zero (positive here)
  if (h) *h = (int32_t)(long)((double)H0 * s);
  if (w) *w = (int32_t)(long)((double)W0 * s);
  if (im_scale) *im_scale = s;
  return MPN_OK;
}

// the sizes of N images and the canvas H = max h_i, W = max w_i (host only)
int mpn_get_images_batch_size_impl(int32_t N, const int32_t *H0, const int32_t *W0, double scale, double max_size, int32_t *h,
                                   int32_t *w, double *im_scale, int32_t *H, int32_t *W) {
  if (N < 1 || N > MPN_MAX_BATCH || !H0 || !W0) return MPN_ERR_ARG;
  int32_t Hm = 0, Wm = 0;
  for (int i = 0; i < N; ++i) {
    int32_t hi = 0, wi = 0; double si = 0;
    if (mpn_get_images_size_impl(H0[i], W0[i], scale, max_size, &hi, &wi, &si) != MPN_OK || hi <= 0 || wi <= 0) return MPN_ERR_ARG;
    if (h) h[i] = hi;
    if (w) w[i] = wi;
    if (im_scale) im_scale[i] = si;
    Hm = hi > Hm ? hi : Hm; Wm = wi > Wm ? wi : Wm;
  }
  if (H) *H = Hm;
  if (W) *W = Wm;
  return MPN_OK;
}

// host-side check of a transformer (nothing enqueued): swap entries are 1-based channel numbers
static int image_transform_check(mpn_ctx *ctx, const mpn_image_transform *tf) {
  MPN_CHECK_ARG(ctx, tf, "getImages: transformer missing");
  for (int c = 0; c < 3; ++c)
    MPN_CHECK_ARG(ctx, tf->swap[c] >= 1 && tf->swap[c] <= 3, "ImageTransformer: swap entries are 1-based channel numbers");
  return MPN_OK;
}

// every host-side check of a batched getImages before anything is enqueued -> the scaled sizes (h, w, im_scale arrays of N;
// im_scale may be null), the canvas and the packed source bytes
int mpn_get_images_batch_check(mpn_ctx *ctx, int32_t N, const int32_t *H0, const int32_t *W0, const mpn_image_transform *tf, double scale,
                               double max_size, int32_t *h, int32_t *w, double *im_scale, int32_t &H, int32_t &W, size_t &in_bytes) {
  MPN_CHECK_ARG(ctx, N >= 1 && N <= MPN_MAX_BATCH, "batch size N must be in 1..MPN_MAX_BATCH");
  MPN_CHECK_ARG(ctx, H0 && W0, "getImages: H0 / W0 missing");
  for (int i = 0; i < N; ++i) MPN_CHECK_ARG(ctx, H0[i] > 0 && W0[i] > 0, "every raw image needs H0, W0 > 0");
  MPN_CHECK_ARG(ctx, mpn_get_images_batch_size_impl(N, H0, W0, scale, max_size, h, w, im_scale, &H, &W) == MPN_OK, "bad scale / max_size");
  MPN_CHECK_ARG(ctx, H <= 65535, "getImages: canvas height above 65535");
  MPN_TRY(image_transform_check(ctx, tf));
  in_bytes = 0;
  for (int i = 0; i < N; ++i) in_bytes += 3 * (size_t)H0[i] * W0[i];
  return MPN_OK;
}

// N images (fp32 3 x H0 x W0 planes or uint8 H0 x W0 x 3 bytes, back to back) of scaled sizes h[i] x w[i] -> the N x 3 x H x W
// canvas, in one launch
int mpn_get_images_batch_launch(mpn_ctx *ctx, const float *im_dev, const uint8_t *im_u8_dev, int32_t N, const int32_t *H0,
                                const int32_t *W0, const int32_t *h, const int32_t *w, int32_t H, int32_t W,
                                const mpn_image_transform *tf, float *out_dev) {
  MpnProfScope prof_scope__(ctx, MPN_CAT_ELTWISE);
  MPN_CHECK_ARG(ctx, (im_dev || im_u8_dev) && out_dev && tf && H0 && W0 && h && w, "getImages: buffers missing");
  MPN_CHECK_ARG(ctx, N >= 1 && N <= MPN_MAX_BATCH, "getImages: batch size N must be in 1..MPN_MAX_BATCH");
  MPN_CHECK_ARG(ctx, H > 0 && W > 0 && H <= 65535, "getImages: bad sizes");
  MPN_TRY(image_transform_check(ctx, tf));
  mpn_img::ImageBatch B;
  memset(&B, 0, sizeof B);
  B.n = N; B.H = H; B.W = W;
  int64_t off = 0;
  for (int i = 0; i < N; ++i) {
    MPN_CHECK_ARG(ctx, H0[i] > 0 && W0[i] > 0 && h[i] > 0 && w[i] > 0 && h[i] <= H && w[i] <= W, "getImages: bad sizes");
    mpn_img::BatchImage &b = B.img[i];
    b.src_off = off; b.H0 = H0[i]; b.W0 = W0[i]; b.h = h[i]; b.w = w[i];
    b.sx = mpn_img::axis_scale(W0[i], w[i]); b.sy = mpn_img::axis_scale(H0[i], h[i]);
    off += 3 * (int64_t)H0[i] * W0[i];
  }
  mpn_img::TransformedImage &I = B.I;
  I.im = im_dev; I.im_u8 = im_u8_dev; I.lut = nullptr;
  if (im_u8_dev) {     // byte -> float table: the 256 correctly rounded quotients b / 255.0f, divided once on the host (IEEE: same bits)
    if (!ctx->u8_lut_dev) {
      static float tab[256];
      static const bool init = [] { for (int b = 0; b < 256; ++b) tab[b] = (float)b / 255.0f; return true; }();
      (void)init;
      MPN_CUDA(ctx, cudaMalloc((void **)&ctx->u8_lut_dev, sizeof(tab)));
      MPN_CUDA(ctx, cudaMemcpyAsync(ctx->u8_lut_dev, tab, sizeof(tab), cudaMemcpyHostToDevice, ctx->stream));
    }
    I.lut = ctx->u8_lut_dev;
  }
  for (int c = 0; c < 3; ++c) {
    I.t.src_chan[c] = tf->swap[c] - 1;
    I.t.neg_mean[c] = (float)(-(double)tf->mean[c]);
    I.t.std[c] = tf->std[c];
  }
  I.t.has_scale = tf->scale != 1.0f;
  I.t.scale = tf->scale;
  I.t.has_std = tf->has_std != 0;
  dim3 grid((unsigned)((W + 255) / 256), (unsigned)H, 3u * (unsigned)N);
  get_images_kernel<<<grid, 256, 0, ctx->stream>>>(B, out_dev);
  MPN_LAUNCHED(ctx);
  return MPN_OK;
}

int mpn_get_images_launch(mpn_ctx *ctx, const float *im_dev, int32_t H0, int32_t W0, const mpn_image_transform *tf,
                          int32_t h, int32_t w, float *out_dev) {
  return mpn_get_images_batch_launch(ctx, im_dev, nullptr, 1, &H0, &W0, &h, &w, h, w, tf, out_dev);
}
int mpn_get_images_u8_launch(mpn_ctx *ctx, const uint8_t *im_hwc_dev, int32_t H0, int32_t W0, const mpn_image_transform *tf,
                             int32_t h, int32_t w, float *out_dev) {
  return mpn_get_images_batch_launch(ctx, nullptr, im_hwc_dev, 1, &H0, &W0, &h, &w, h, w, tf, out_dev);
}
