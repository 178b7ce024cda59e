// TEST INFRASTRUCTURE: host build of the batched getImages element function (mpn_img::batch_pixel in
// multipathnet_b200/csrc/image_scale.cuh), filled the way mpn_get_images_batch_launch fills its kernel parameters, so the
// CPU suite can run per canvas element what get_images_kernel runs. tests/test_batch_raw_cpu.py compiles it with
// -ffp-contract=off (the device side uses *_rn intrinsics). Not linked into the product.
#include "../multipathnet_b200/csrc/image_scale.cuh"

// ims: N uint8 H0[i] x W0[i] x 3 images back to back; h / w: their scaled sizes; out: N x 3 x H x W
extern "C" int hd_get_images_batch_u8(const unsigned char *ims, int N, const int *H0, const int *W0, const int *h, const int *w, int H,
                                      int W, const int *swap /* 1-based */, float scale, const float *mean, const float *std /* or NULL */,
                                      float *out) {
  if (N < 1 || N > mpn_img::kMaxBatchImages) return -1;
  static float lut[256];
  for (int b = 0; b < 256; ++b) lut[b] = (float)b / 255.0f;
  static mpn_img::ImageBatch B;       // ~2 KB, as the kernel's parameter block
  B = mpn_img::ImageBatch();
  B.n = N; B.H = H; B.W = W;
  long long off = 0;
  for (int i = 0; i < N; ++i) {
    mpn_img::BatchImage &b = B.img[i];
    b.src_off = off; b.H0 = H0[i]; b.W0 = W0[i]; b.h = h[i]; b.w = w[i];
    b.sx = mpn_img::axis_scale(W0[i], w[i]); b.sy = mpn_img::axis_scale(H0[i], h[i]);
    off += 3LL * H0[i] * W0[i];
  }
  mpn_img::TransformedImage &I = B.I;
  I.im = nullptr; I.im_u8 = ims; I.lut = lut; I.H0 = 0; I.W0 = 0;
  for (int c = 0; c < 3; ++c) {
    I.t.src_chan[c] = swap[c] - 1;
    I.t.neg_mean[c] = (float)(-(double)mean[c]);
    I.t.std[c] = std ? std[c] : 1.0f;
  }
  I.t.has_scale = scale != 1.0f;
  I.t.scale = scale;
  I.t.has_std = std != nullptr;
  for (int n = 0; n < N; ++n)
    for (int c = 0; c < 3; ++c)
      for (int y = 0; y < H; ++y)
        for (int x = 0; x < W; ++x) out[(((long)n * 3 + c) * H + y) * W + x] = mpn_img::batch_pixel(B, n, c, y, x);
  return 0;
}
