// getImages on the device (SURVEY 8f-1): ImageTransformer + image.scale, one output pixel at a time.
//
// Reference: ImageDetect.lua:22-52 (getImages: transformer, im_scale, image.scale(im, w, h)),
// modules/ImageTransformer.lua:19-33 (channel swap, x scale, - mean, / std, in that order, fp32).
// `image.scale` lives in the third-party torch `image` package (absent from /root/reference, luarocks scm, no pin):
// its default 'bilinear' mode is restated here from image/generic/image.c (scaleBilinear -> scaleLinear_rowcol) as
// recalled -- PARITY UNPINNED:
//   * separable: every source row is resampled to the new width first (fp32 temporary), then every column of that
//     temporary to the new height;
//   * a longer axis (dst_len > src_len) is linear interpolation with corners aligned: scale = (src_len-1)/(dst_len-1),
//     s = di*scale, out = (1-frac)*src[int(s)] + frac*src[int(s)+1], the last sample copies src[src_len-1];
//   * a shorter axis (dst_len < src_len) is an area average: scale = src_len/dst_len, the window [di*scale, (di+1)*scale)
//     with fractional end weights, out = acc / n;
//   * an equal axis is a copy.
// Everything below is fp32 with the operation order of that C code and no fused multiply-add (explicit *_rn on the
// device; the host build of this header, oracle/hd_shim.cpp, is compiled with -ffp-contract=off), so that the fused
// single-pass kernel reproduces the two-pass original bit for bit: a temporary sample is recomputed, never changed.
//
// The functions are __host__ __device__ so that the CPU suite can run the very arithmetic the kernel runs
// (tests/test_getimages_cpu.py through oracle/hd_shim.cpp) against the independent two-pass restatement in
// oracle/mpn_oracle.c.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define MPN_HD __host__ __device__ __forceinline__
#else
#define MPN_HD inline
#endif

namespace mpn_img {

MPN_HD float fmul(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fmul_rn(a, b);
#else
  return a * b;
#endif
}
MPN_HD float fadd(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fadd_rn(a, b);
#else
  return a + b;
#endif
}
MPN_HD float fsub(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fsub_rn(a, b);
#else
  return a - b;
#endif
}
MPN_HD float fdiv(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fdiv_rn(a, b);
#else
  return a / b;
#endif
}

// fbcoco.ImageTransformer(mean, std, scale, swap) (ImageTransformer.lua:11-17), flattened for the kernel
struct Transform {
  int32_t src_chan[3];   // 0-based source channel of output channel c (swap, :21); identity = {0,1,2}
  int32_t has_scale;     // self.scale ~= 1 (:22)
  float scale;
  float neg_mean[3];     // I[i]:add(-mean[i]) (:26)
  int32_t has_std;       // (:27)
  float std[3];
};

// one sample of the transformed image (before resizing)
struct TransformedImage {
  const float *im;       // 3 x H0 x W0 fp32, RGB in [0,1] (loaders/loader.lua:79), or null with:
  const uint8_t *im_u8;  // H0 x W0 x 3 bytes, interleaved RGB as a decoder hands them over; the value is byte / 255 in fp32
                         // (what image.load(path, 3, 'float') returns), one IEEE division per sample
  const float *lut;      // optional: lut[b] = (float)b / 255.0f for b = 0..255, the SAME correctly rounded quotients, computed once
                         // (the kernel spent a third of its instructions in four IEEE divisions per output pixel, and a zero byte
                         // sends div.rn down its slow path); null = divide
  int32_t H0, W0;
  Transform t;
  MPN_HD float byte_value(uint8_t b) const {
#if defined(__CUDA_ARCH__)
    return lut ? __ldg(lut + b) : fdiv((float)b, 255.0f);
#else
    return lut ? lut[b] : fdiv((float)b, 255.0f);
#endif
  }
  MPN_HD float at(int c, int y, int x) const {      // selects, not indexing: the struct stays in kernel-parameter space
    const int sc = c == 0 ? t.src_chan[0] : (c == 1 ? t.src_chan[1] : t.src_chan[2]);
    float v = im ? im[((int64_t)sc * H0 + y) * W0 + x] : byte_value(im_u8[((int64_t)y * W0 + x) * 3 + sc]);
    if (t.has_scale) v = fmul(v, t.scale);
    v = fadd(v, c == 0 ? t.neg_mean[0] : (c == 1 ? t.neg_mean[1] : t.neg_mean[2]));
    if (t.has_std) v = fdiv(v, c == 0 ? t.std[0] : (c == 1 ? t.std[1] : t.std[2]));
    return v;
  }
};

// the step of a 1-D resample src_len -> dst_len (one IEEE division; the kernel gets it precomputed on the host, same bits)
MPN_HD float axis_scale(int src_len, int dst_len) {
  if (dst_len > src_len) return (src_len == 1) ? 0.0f : fdiv((float)(src_len - 1), (float)(dst_len - 1));
  if (dst_len < src_len) return fdiv((float)src_len, (float)dst_len);
  return 1.0f;
}

// one output sample di of a 1-D resample src_len -> dst_len; get(i) reads source sample i; scale = axis_scale(src_len, dst_len)
template <class Get>
MPN_HD float scale1d(int src_len, int dst_len, int di, const Get &get, const float scale) {
  if (dst_len > src_len) {
    if (src_len == 1 || di == dst_len - 1) return get(src_len - 1);
    float sf = fmul((float)di, scale);
    int si = (int)sf;
    sf = fsub(sf, (float)si);
    if (si >= src_len - 1) return get(src_len - 1);           // rounding guard: never read past the last sample
    return fadd(fmul(fsub(1.0f, sf), get(si)), fmul(sf, get(si + 1)));
  }
  if (dst_len < src_len) {
    float s0f = fmul((float)di, scale);
    int s0 = (int)s0f;
    s0f = fsub(s0f, (float)s0);
    float s1f = fmul((float)(di + 1), scale);
    int s1 = (int)s1f;
    s1f = fsub(s1f, (float)s1);
    if (s0 > src_len - 1) s0 = src_len - 1;
    float acc = fmul(fsub(1.0f, s0f), get(s0));
    float n = fsub(1.0f, s0f);
    for (int s = s0 + 1; s < s1 && s < src_len; ++s) {
      acc = fadd(acc, get(s));
      n = fadd(n, 1.0f);
    }
    if (s1 < src_len) {
      acc = fadd(acc, fmul(s1f, get(s1)));
      n = fadd(n, s1f);
    }
    return fdiv(acc, n);
  }
  return get(di);
}
template <class Get>
MPN_HD float scale1d(int src_len, int dst_len, int di, const Get &get) { return scale1d(src_len, dst_len, di, get, axis_scale(src_len, dst_len)); }

struct RowGet {               // source row y of channel c, sampled along x
  const TransformedImage *I;
  int c, y;
  MPN_HD float operator()(int x) const { return I->at(c, y, x); }
};
struct TmpColGet {            // column x of the width-resampled temporary (H0 x w), sampled along y
  const TransformedImage *I;
  int c, x, w;
  float sx;                   // axis_scale(W0, w)
  MPN_HD float operator()(int y) const {
    RowGet r{I, c, y};
    return scale1d(I->W0, w, x, r, sx);
  }
};

// pixel (c, y, x) of image.scale(transformer(im), w, h); sx / sy = axis_scale(W0, w) / axis_scale(H0, h)
MPN_HD float scaled_pixel(const TransformedImage &I, int h, int w, int c, int y, int x, float sx, float sy) {
  TmpColGet col{&I, c, x, w, sx};
  return scale1d(I.H0, h, y, col, sy);
}
MPN_HD float scaled_pixel(const TransformedImage &I, int h, int w, int c, int y, int x) {
  return scaled_pixel(I, h, w, c, y, x, axis_scale(I.W0, w), axis_scale(I.H0, h));
}

// getImages of N images into one zero-padded N x 3 x H x W canvas (ImageDetect.lua:44-50: images:resize(n,3,maxH,maxW):zero(),
// each image copied top-left). The sources lie back to back: image n starts src_off elements after the shared base pointer
// (3*H0*W0 per image, bytes for the uint8 source, floats for the fp32 one).
enum { kMaxBatchImages = 64 };       // MPN_MAX_BATCH (include/mpn_abi.h)
struct BatchImage {
  int64_t src_off;
  int32_t H0, W0;        // original size
  int32_t h, w;          // scaled size (mpn_get_images_size)
  float sx, sy;          // axis_scale(W0, w), axis_scale(H0, h), divided on the host
};
struct ImageBatch {
  TransformedImage I;    // base pointer(s), byte table and transformer shared by all images; I.H0 / I.W0 unused
  int32_t n, H, W;       // images, canvas
  BatchImage img[kMaxBatchImages];
};

// element (n, c, y, x) of the canvas: image n's scaled pixel inside [0, h) x [0, w), +0.0f elsewhere
MPN_HD float batch_pixel(const ImageBatch &B, int n, int c, int y, int x) {
  const BatchImage &b = B.img[n];
  if (y >= b.h || x >= b.w) return 0.0f;
  TransformedImage I = B.I;
  I.H0 = b.H0; I.W0 = b.W0;
  if (I.im) I.im += b.src_off;
  else I.im_u8 += b.src_off;
  return scaled_pixel(I, b.h, b.w, c, y, x, b.sx, b.sy);
}

}  // namespace mpn_img
