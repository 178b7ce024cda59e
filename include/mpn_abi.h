/* ============================================================================
 * mpn_abi.h — C ABI of libmpn_b200.so: the drop-in boundary for the
 * multipathnet detection forward hot path on B200 (sm_100a).
 *
 * Plain C declarations only (no macros in prototypes, no torch/TH types) so the
 * block between MPN_CDEF_BEGIN/END can be pasted verbatim into LuaJIT
 * `ffi.cdef` (lua/mpn_ffi.lua does exactly that) and is what Python loads via
 * ctypes (multipathnet_b200/_lib.py). Every entry point names the reference
 * interface it replaces (paths relative to facebookresearch/multipathnet).
 *
 * Conventions
 *  - every function returns 0 on success, <0 on error; text via mpn_last_error.
 *    Nothing exits, throws, or longjmps across the boundary.
 *  - `*_dev` pointers are device pointers on the ctx's device; others are host
 *    pointers. The caller owns all I/O buffers; the library owns ctx/model only.
 *  - calls run on the ctx's stream; entry points taking/returning HOST buffers
 *    are synchronous (like the reference's blocking :float()/:cuda() copies),
 *    `_dev` entry points are stream-ordered and asynchronous.
 *  - boxes are 1-based pixel coordinates [x1,y1,x2,y2]; ROI rows are
 *    [batch_idx(1-based), x1, y1, x2, y2] (ImageDetect.lua:66-70).
 *  - no global mutable state: one mpn_ctx per (thread, device)
 *    (test_runner.lua:55-66 runs one replica per thread/GPU).
 * ==========================================================================*/
#ifndef MPN_ABI_H
#define MPN_ABI_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif
/* MPN_CDEF_BEGIN */

typedef struct mpn_ctx mpn_ctx;
typedef struct mpn_model mpn_model;

/* ---- context ------------------------------------------------------------- */
/* device: CUDA ordinal. cuda_stream: a cudaStream_t, or NULL for the legacy
 * default stream (what cutorch uses unless cutorch.setStream was called).   */
int mpn_ctx_create(int device, void *cuda_stream, mpn_ctx **out);
/* A context on a stream of its own (non-blocking, created and destroyed with the ctx; priority as cudaStreamCreateWithPriority,
 * clamped to the device's range, 0 = default): for SEVERAL model replicas on one GPU. The reference runs one model replica per
 * donkey thread (test_runner.lua:55-66); with K threads per GPU, each on its own ctx / stream, the layer-boundary and NMS-chain
 * bubbles of one replica are filled by the kernels of the others (+8 % proposals/s at K = 2 on cfg 2). Work of different
 * contexts is unordered; mpn_ctx_wait_ctx(ctx, other) makes everything enqueued on `ctx` afterwards wait for what `other` has
 * enqueued so far (the join before the end-of-run gather). mpn_ctx_stream returns the cudaStream_t (interop with the caller's
 * own kernels / events). */
int mpn_ctx_create_stream(int device, int priority, mpn_ctx **out);
void *mpn_ctx_stream(const mpn_ctx *ctx);
int mpn_ctx_wait_ctx(mpn_ctx *ctx, mpn_ctx *other);
void mpn_ctx_destroy(mpn_ctx *ctx);
const char *mpn_last_error(const mpn_ctx *ctx);   /* ctx may be NULL: last create error */
int mpn_ctx_synchronize(mpn_ctx *ctx);
/* number of kernels THIS library launched on ctx since creation (bench.py's gpu_launches) */
int64_t mpn_ctx_launch_count(const mpn_ctx *ctx);
const char *mpn_version(void);
/* run-time knobs of the product kernels, so that tests can cover every variant in one process; value < 0 restores the
 * default (the environment variable of the same meaning, else the built-in choice). Names:
 *   "fc_w16"          numerics of the big per-ROI Linears (fc6 / fc7: K >= 2048, >= 1024 outputs), read when a model plans
 *                     its heads: 1 = weight as ONE fp16 plane scaled by a power of two, two tensor-core products per
 *                     MAC (A_hi x W + A_lo x W); 0 = the three-product bf16 split every other layer uses. Unset: 1 for
 *                     single-tower graphs (Fast R-CNN: 4-5e-4 on the scores at full size), 0 for multi-tower graphs
 *                     (MultiPathNet measured 2.3e-3 with it: outside the 1e-3 contract). Environment: MPN_FC_W16.
 *   "roi_impl"        fused Foveal + ROI pooling kernel: 0 = roi_pool_cluster_kernel (default: 4-CTA clusters, the
 *                     L2 norm reduced over distributed shared memory), 1 = the round-1 kernel (one block stages a
 *                     normalised level's whole vector), 2 = the round-1 two-pass variant (sum-of-squares pre-pass +
 *                     unstaged writing pass), 3 = the cluster kernel exchanging its partial sums through
 *                     barrier.cluster instead of st.async, 4 = roi_pool_bulk_kernel (the pyramid blocks arrive in
 *                     shared-memory slots by cp.async.bulk), 5 = roi_pool_ring_kernel (one persistent CTA per SM: a
 *                     producer warp keeps a ring of bulk-copy stages full, 16 consumer warps drain it).
 *                     Environment: MPN_ROI_IMPL.
 *   "roi_norm_split"  older spelling: 1 selects roi_impl 2, 0 selects roi_impl 1 (MPN_ROI_NORM_SPLIT).          */
int mpn_ctx_set_option(mpn_ctx *ctx, const char *name, int64_t value);
/* per-category kernel timing for roofline reporting: between begin and end every launch group is
 * bracketed by CUDA events on the ctx stream. ms_by_cat[6] = {conv/GEMM tcgen05, first-layer direct conv,
 * fused ROI pooling, NMS, elementwise glue, max/avg pooling}; launches_by_cat likewise (may be NULL). */
int mpn_ctx_profile_begin(mpn_ctx *ctx);
int mpn_ctx_profile_end(mpn_ctx *ctx, double *ms_by_cat, int64_t *launches_by_cat);
/* in-kernel timeline of the tcgen05 launches (diagnostics, tools/timeline.py): between begin and end every tensor-core
 * launch i records %globaltimer stamps, min over CTAs in stamps_min[4i..]: {kernel entry, dependency wait passed, first
 * MMA issued, -}, max over CTAs in stamps_max[4i..]: {last MMA issued, last epilogue finished, kernel exit, -} (ns). */
int mpn_ctx_timeline_begin(mpn_ctx *ctx, int32_t max_launches);
int mpn_ctx_timeline_end(mpn_ctx *ctx, uint64_t *stamps_min, uint64_t *stamps_max, int32_t *n_launches);

/* ---- NMS: replaces utils.nms -> nms.c:NMS (utils.lua:29-33, nms.c:59-108) --
 * scored_boxes: N x 5 [x1,y1,x2,y2,score]. Writes the kept ROW INDICES
 * (0-based, selection order = the order nms.c emits its kept rows) into
 * keep_idx (capacity N) and the count into *n_keep. Bit-exact vs nms.c,
 * including its tie behaviour. Host buffers, synchronous.                   */
int mpn_nms(mpn_ctx *ctx, const float *scored_boxes, int64_t N, float thr,
            int32_t *keep_idx, int64_t *n_keep);
/* Batched form (one launch set for all classes of an image, Tester_FRCNN.lua:106-117):
 * segment s covers rows [seg_offsets[s], seg_offsets[s+1]) of scored_boxes;
 * keep_idx is written at the same offsets (indices local to the segment),
 * keep_counts[s] = number kept. Host buffers, synchronous.                  */
int mpn_nms_batched(mpn_ctx *ctx, const float *scored_boxes, const int64_t *seg_offsets,
                    int64_t nseg, float thr, int32_t *keep_idx, int64_t *keep_counts);
/* Same, device buffers, stream-ordered (seg_offsets stays on the host).     */
int mpn_nms_batched_dev(mpn_ctx *ctx, const float *scored_boxes_dev, const int64_t *seg_offsets,
                        int64_t nseg, float thr, int32_t *keep_idx_dev, int32_t *keep_counts_dev);
/* replaces utils.nms_dense (utils.lua:402-462, used by demo.lua:85): 0-based
 * original indices in descending-score order; ties broken by ascending index. */
int mpn_nms_dense(mpn_ctx *ctx, const float *scored_boxes, int64_t N, float thr,
                  int32_t *pick_idx, int64_t *n_pick);
/* replaces utils.bbox_vote -> nms.c:bbox_vote (utils.lua:35-39, nms.c:110-142) */
int mpn_bbox_vote(mpn_ctx *ctx, const float *nms_boxes, int64_t K, const float *scored_boxes,
                  int64_t N, float thr, float *res);

/* ---- region modules ------------------------------------------------------ */
/* nn.Foveal:updateOutput (modules/Foveal.lua:15-44): R x 5 -> 4R x 5, the four
 * regions of ROI i consecutive; fp64 arithmetic rounded once to fp32.       */
int mpn_foveal(mpn_ctx *ctx, const float *rois, int64_t R, float *out);
/* nn.ContextRegion(scale):updateOutput (modules/ContextRegion.lua:14-32)     */
int mpn_context_region(mpn_ctx *ctx, const float *rois, int64_t R, float scale, float *out);
/* nn.BBoxNorm:updateOutput, evaluate mode (modules/BBoxNorm.lua:18-32): in place */
int mpn_bbox_norm(mpn_ctx *ctx, float *deltas, int64_t R, int64_t C4, const float *mean4,
                  const float *std4);
/* the three modules on DEVICE buffers (CudaTensors), stream-ordered, no copies: the reference's Foveal takes its input to the
 * host and back on every forward (Foveal.lua:21-22,42). mean4 / std4 stay host pointers (4 floats each).                */
int mpn_foveal_dev(mpn_ctx *ctx, const float *rois_dev, int64_t R, float *out_dev);
int mpn_context_region_dev(mpn_ctx *ctx, const float *rois_dev, int64_t R, float scale, float *out_dev);
int mpn_bbox_norm_dev(mpn_ctx *ctx, float *deltas_dev, int64_t R, int64_t C4, const float *mean4,
                      const float *std4);
/* utils.convertFrom tensor branch applied per class block of 4
 * (ImageDetect.lua:183-185, utils.lua:226-246): deltas R x 4C, boxes R x 4.   */
int mpn_bbox_decode(mpn_ctx *ctx, const float *deltas, const float *boxes, int64_t R, int64_t C,
                    float *out);

/* ---- inn.ROIPooling(W,H,scale):updateOutput {data, rois} ------------------
 * (call sites vgg.lua:28, alexnet.lua:23, resnet.lua:48, model_utils.lua:215)
 * fmap N x C x H x W fp32 (NCHW as Torch holds it), rois R x 5, out
 * R x C x PH x PW, argmax (R*C*PH*PW int32, flat h*W+w or -1) may be NULL.
 * variant: 1 = Caffe port (end inclusive), 2 = imagine-nn v2 (default).     */
int mpn_roi_pool(mpn_ctx *ctx, const float *fmap, int64_t N, int64_t C, int64_t H, int64_t W,
                 const float *rois, int64_t R, int32_t PW, int32_t PH, float spatial_scale,
                 int32_t variant, float *out, int32_t *argmax);
int mpn_roi_pool_dev(mpn_ctx *ctx, const float *fmap_dev, int64_t N, int64_t C, int64_t H,
                     int64_t W, const float *rois_dev, int64_t R, int32_t PW, int32_t PH,
                     float spatial_scale, int32_t variant, float *out_dev, int32_t *argmax_dev);

/* ---- model: the nn.Sequential graphs of models/{vgg,multipathnet,resnet}.lua
 * described as data. Layers operate on numbered tensor slots; slot 0 of the
 * trunk is the input image (1 x 3 x H x W fp32, post-transformer).          */
enum {
  MPN_LAYER_CONV = 1,       /* conv kh x kw, stride, pad, + bias [+ residual] [+ ReLU]; a Linear is a 1x1 conv on a 1x1 map */
  MPN_LAYER_MAXPOOL = 2,    /* k x k, stride, pad, ceil_mode */
  MPN_LAYER_AVGPOOL = 3,    /* global average over H x W (ResNet avgpool 7) */
  MPN_LAYER_FLATTEN = 4     /* (H,W,C) -> 1 x 1 x (H*W*C); reference order (c,ph,pw) is honoured by permuting the next weight */
};
typedef struct mpn_layer {
  int32_t kind;
  int32_t in_slot, out_slot;
  int32_t cin, cout, kh, kw, stride, pad;
  int32_t relu;             /* 1: ReLU fused after bias(+residual) */
  int32_t residual_slot;    /* slot added before ReLU, or -1 */
  int32_t ceil_mode;        /* pooling only */
  int32_t weight, bias;     /* indices into weights[], -1 = none; conv weight is Cout x Cin x kh x kw (Torch layout) */
} mpn_layer;

typedef struct mpn_tower {   /* one region tower of multipathnet.lua:73-113, or THE head of vgg/resnet */
  int32_t region;           /* 0 = the ROI itself, 1..3 = Foveal regions x1.5, x2, x4 (Foveal.lua:36-39) */
  int32_t n_levels;         /* 1..3 pooled trunk taps, channel-concat order (model_utils.lua:229-235) */
  int32_t level_slot[3];    /* trunk slot of each level */
  float   level_scale[3];   /* spatial scale of each level (1/16, 1/8, 1/4) */
  int32_t pooled_w, pooled_h;
  int32_t normalize;        /* 1: L2-normalise each level then x1000 (model_utils.lua:217-220,240) */
  int32_t n_layers;         /* per-ROI layers applied to the pooled R x PH x PW x C tensor (slot 0) */
  int32_t first_layer;      /* index into the model's tower_layers[] array */
  int32_t out_slot;         /* tower-local slot holding the R x 1 x 1 x F result */
} mpn_tower;

typedef struct mpn_head {    /* Linear over a column range of the towers' concat (multipathnet.lua:115-117) */
  int32_t col_begin, col_len;
  int32_t cout;
  int32_t weight, bias;
} mpn_head;

typedef struct mpn_model_desc {
  int32_t n_trunk_layers;  const mpn_layer *trunk_layers;
  int32_t n_towers;        const mpn_tower *towers;
  int32_t n_tower_layers;  const mpn_layer *tower_layers;
  int32_t n_cls_heads;     const mpn_head *cls_heads;   /* >1: integral head, eval = mean of softmaxes (model_utils.lua:296-313) */
  mpn_head bbox_head;
  int32_t num_classes;     /* C incl. background */
  int32_t roi_variant;     /* 1 or 2, see mpn_roi_pool */
  int32_t no_softmax;      /* model.noSoftMax (ImageDetect.lua:189): scores are already probabilities */
  int32_t has_bbox_norm;   /* nn.BBoxNorm appended (model_utils.lua:176-182) */
  float bbox_mean[4], bbox_std[4];
  int32_t max_rois;        /* capacity to allocate for */
  int32_t max_h, max_w;    /* largest scaled image */
} mpn_model_desc;

/* weights[i] are HOST fp32 arrays in Torch layout with n_elem[i] elements; they are
 * copied/re-laid-out at create, nothing is retained.                         */
int mpn_model_create(mpn_ctx *ctx, const mpn_model_desc *desc, const float *const *weights,
                     const int64_t *n_elem, int32_t n_weights, mpn_model **out);
void mpn_model_destroy(mpn_model *m);

/* model:get(1):forward — the conv trunk, once per image (ImageDetect.lua:107-108).
 * image: 3 x H x W fp32 host (or device with _dev), already transformed+scaled. */
int mpn_model_trunk(mpn_model *m, const float *image, int32_t H, int32_t W);
int mpn_model_trunk_dev(mpn_model *m, const float *image_dev, int32_t H, int32_t W);
/* model:get(1):forward on a batch: images N x 3 x H x W (post-transformer, one size: the caller pads as getImages does,
 * zeros after the transformer, ImageDetect.lua:44-50), 1 <= N <= MPN_MAX_BATCH. Later mpn_model_heads* / get_pooled /
 * get_trunk_slot calls see all N images; ROI rows pick their image with column 0 (1-based), and a row naming an image
 * outside [1, N] fails the call (host entries) or raises the ctx's device flag (_dev entries: the next synchronous call
 * or mpn_ctx_synchronize fails). N = 1 is exactly mpn_model_trunk(_dev).                                             */
enum { MPN_MAX_BATCH = 64 };
int mpn_model_trunk_batch_dev(mpn_model *m, const float *images_dev, int32_t N, int32_t H, int32_t W);
int mpn_model_trunk_batch(mpn_model *m, const float *images, int32_t N, int32_t H, int32_t W);
/* ---- getImages on the device (SURVEY 8f-1): ImageDetect.lua:22-52 + modules/ImageTransformer.lua:19-33 ----------
 * fbcoco.ImageTransformer(mean, std, scale, swap) as plain data: out[c] = (im[swap[c]] * scale - mean[c]) / std[c],
 * each step fp32 in that order, `* scale` skipped when scale == 1, `/ std` when has_std == 0 (RossTransformer:
 * swap {3,2,1}, scale 255, Ross' BGR means, no std; ImagenetTransformer: swap {1,2,3}, scale 1, mean + std;
 * model_utils.lua:138-155).                                                                                  */
typedef struct mpn_image_transform {
  int32_t swap[3];   /* 1-based source channel of each output channel */
  float scale;
  float mean[3];
  float std[3];
  int32_t has_std;
} mpn_image_transform;
/* host-only (no GPU): the size getImages scales a H0 x W0 image to for the single test scale (`scale`, `max_size` as
 * ImageDetect.lua:17-18) and the im_scale it returns: im_scale = scale / min side, capped so that
 * round(im_scale * max side) <= max_size; h = trunc(H0 * im_scale), w = trunc(W0 * im_scale) (:31-39). */
int mpn_get_images_size(int32_t H0, int32_t W0, double scale, double max_size, int32_t *h, int32_t *w, double *im_scale);
/* transformer + image.scale(im, w, h) ('bilinear', the third-party `image` package: parity unpinned, see
 * csrc/image_scale.cuh) in one kernel. im: 3 x H0 x W0 fp32 RGB in [0,1] (loaders/loader.lua:79), out: 3 x h x w.
 * Host buffers, synchronous; _dev: device buffers, stream-ordered. */
int mpn_get_images(mpn_ctx *ctx, const float *im, int32_t H0, int32_t W0, const mpn_image_transform *tf,
                   int32_t h, int32_t w, float *out);
int mpn_get_images_dev(mpn_ctx *ctx, const float *im_dev, int32_t H0, int32_t W0, const mpn_image_transform *tf,
                       int32_t h, int32_t w, float *out_dev);
/* Same from the decoder's bytes: im_hwc H0 x W0 x 3 uint8, interleaved RGB; the sample value is byte / 255 in fp32 (what
 * image.load(path, 3, 'float') hands to the transformer): a quarter of the bytes to move over the bus. */
int mpn_get_images_u8(mpn_ctx *ctx, const uint8_t *im_hwc, int32_t H0, int32_t W0, const mpn_image_transform *tf,
                      int32_t h, int32_t w, float *out);
int mpn_get_images_u8_dev(mpn_ctx *ctx, const uint8_t *im_hwc_dev, int32_t H0, int32_t W0, const mpn_image_transform *tf,
                          int32_t h, int32_t w, float *out_dev);
/* host-only (no GPU): getImages sizes of N images (mpn_get_images_size of each: h, w, im_scale arrays of N, any may be
 * NULL) and the padded canvas H = max h_i, W = max w_i. Fails for N outside 1..MPN_MAX_BATCH or a size <= 0. */
int mpn_get_images_batch_size(int32_t N, const int32_t *H0, const int32_t *W0, double scale, double max_size,
                              int32_t *h, int32_t *w, double *im_scale, int32_t *H, int32_t *W);
/* getImages of N raw images into one zero-padded N x 3 x H x W batch (ImageDetect.lua:44-50), in one launch. ims_hwc: the
 * images' bytes back to back, image i H0[i] x W0[i] x 3 interleaved RGB at byte offset sum_{j<i} 3*H0[j]*W0[j]; one
 * transformer for all. Image i's block [0,h_i) x [0,w_i) is exactly what mpn_get_images_u8 gives for it alone, every other
 * element is +0.0f (written by the kernel: out needs no clearing). H, W as mpn_get_images_batch_size, H <= 65535.
 * Host buffers, synchronous; _dev: device buffers, stream-ordered. */
int mpn_get_images_batch_u8(mpn_ctx *ctx, const uint8_t *ims_hwc, int32_t N, const int32_t *H0, const int32_t *W0,
                            const mpn_image_transform *tf, double scale, double max_size, float *out);
int mpn_get_images_batch_u8_dev(mpn_ctx *ctx, const uint8_t *ims_hwc_dev, int32_t N, const int32_t *H0, const int32_t *W0,
                                const mpn_image_transform *tf, double scale, double max_size, float *out_dev);
/* getImages + model:get(1):forward: uploads the RAW image (host), transforms and scales it on the device into the
 * model's image buffer and runs the trunk; *im_scale, *h, *w as mpn_get_images_size. Follow with mpn_model_detect(...,
 * image = NULL, recompute_features = 0) on the cached features. */
int mpn_model_trunk_image(mpn_model *m, const float *im, int32_t H0, int32_t W0, const mpn_image_transform *tf,
                          double scale, double max_size, double *im_scale, int32_t *h, int32_t *w);
/* modules 2..n on cached trunk features (recompute_features=false path,
 * ImageDetect.lua:109-124): rois R x 5 in scaled-image coords. Outputs are the
 * RAW network outputs: cls R x C (logits, or probabilities if no_softmax) and
 * bbox R x 4C (after BBoxNorm if present) = what model:forward returns.      */
int mpn_model_heads(mpn_model *m, const float *rois, int64_t R, float *cls_out, float *bbox_out);
int mpn_model_heads_dev(mpn_model *m, const float *rois_dev, int64_t R, float *cls_out_dev,
                        float *bbox_out_dev);

/* ImageDetect:detect (ImageDetect.lua:156-193) after getImages: trunk (if
 * recompute_features) + heads + convertFrom per class with the ORIGINAL boxes +
 * softmax unless no_softmax. boxes R x 4 original-image coords, im_scale from
 * getImages. scores R x C, bboxes R x 4C (host, synchronous).                */
int mpn_model_detect(mpn_model *m, const float *image, int32_t H, int32_t W, const float *boxes,
                     int64_t R, float im_scale, int32_t recompute_features, float *scores,
                     float *bboxes);
/* detect + Tester_FRCNN:testOne post-processing (Tester_FRCNN.lua:75-78,106-117)
 * in one stream-ordered pass: clamp to [1,W0]x[1,H0], per foreground class
 * gather [box,score] rows with score > score_thresh, NMS at nms_thr.
 * keep_idx: (C-1) x R int32 (row indices into the R proposals, selection order),
 * keep_counts: C-1. scores/bboxes as mpn_model_detect but bboxes are clamped.
 * All pointers host; any of scores/bboxes may be NULL to skip that copy.     */
int mpn_model_detect_nms(mpn_model *m, const float *image, int32_t H, int32_t W,
                         const float *boxes, int64_t R, float im_scale, float W0, float H0,
                         float score_thresh, float nms_thr, float *scores, float *bboxes,
                         int32_t *keep_idx, int32_t *keep_counts);
/* Pipelined form of mpn_model_detect_nms for throughput serving (test_runner.lua keeps one
 * image in flight per donkey thread; here one model keeps two): submit returns at once with a
 * ticket, at most 2 tickets may be outstanding. The host->device copy of a submission runs on
 * its own copy stream and overlaps the kernels of the previous submission, the device->host
 * copy of the results on a third stream. The caller's buffers (pinned memory for real overlap)
 * must stay valid and untouched until mpn_model_detect_nms_wait(ticket) returns; results are
 * bit-identical to the synchronous call.                                       */
int mpn_model_detect_nms_submit(mpn_model *m, const float *image, int32_t H, int32_t W,
                                const float *boxes, int64_t R, float im_scale, float W0, float H0,
                                float score_thresh, float nms_thr, float *scores, float *bboxes,
                                int32_t *keep_idx, int32_t *keep_counts, int32_t *ticket);
/* The same pipeline fed with the RAW image as the decoder leaves it (H0 x W0 x 3 uint8, interleaved RGB): getImages
 * (ImageDetect.lua:22-52: transformer, im_scale rule for `scale` / `max_size`, image.scale) runs on the device in front
 * of the trunk, boxes are original-image coordinates, the clamp is to the original W0 x H0. 0.9 MB cross the bus for a
 * 480 x 640 image instead of the 5.8 MB of its scaled fp32 form. Same ticket protocol as mpn_model_detect_nms_submit. */
int mpn_model_detect_nms_submit_u8(mpn_model *m, const uint8_t *im_hwc, int32_t H0, int32_t W0,
                                   const mpn_image_transform *tf, double scale, double max_size, const float *boxes,
                                   int64_t R, float score_thresh, float nms_thr, float *scores, float *bboxes,
                                   int32_t *keep_idx, int32_t *keep_counts, int32_t *ticket);
/* Pipelined mpn_model_detect_nms_batch from N RAW images of any sizes (packed as mpn_get_images_batch_u8): the packed bytes
 * and the boxes cross the bus on the copy stream, getImages pads the images into one canvas (H = max h_i, W = max w_i) on
 * the device, and the batched trunk, heads and NMS follow. boxes R_total x 4 in each image's ORIGINAL coordinates, image i
 * owning rows [img_offsets[i], img_offsets[i+1]); each image is projected with its own im_scale_i (as float) and clamped
 * to its own W0[i] x H0[i]. Outputs, their layout and the detection sink (N records in image order) as
 * mpn_model_detect_nms_batch. Same ticket protocol and the same two slots as mpn_model_detect_nms_submit(_u8): the kinds
 * may be interleaved, and mpn_model_detect_nms_wait completes either. N = 1 is exactly mpn_model_detect_nms_submit_u8.
 * A canvas that differs from the previous call's re-plans the trunk. Every argument is checked before anything is
 * enqueued: 1 <= N <= MPN_MAX_BATCH, H0, W0 > 0, canvas within the model's max_h x max_w, every R_i >= 1,
 * R_total <= max_rois, swap entries 1..3, pointers present. The synchronous form is submit + wait; device-resident callers
 * compose mpn_get_images_batch_u8_dev with mpn_model_detect_nms_batch_dev. */
int mpn_model_detect_nms_batch_submit_u8(mpn_model *m, const uint8_t *ims_hwc, int32_t N, const int32_t *H0, const int32_t *W0,
                                         const mpn_image_transform *tf, double scale, double max_size,
                                         const float *boxes, const int64_t *img_offsets, float score_thresh, float nms_thr,
                                         float *scores, float *bboxes, int32_t *keep_idx, int32_t *keep_counts, int32_t *ticket);
int mpn_model_detect_nms_wait(mpn_model *m, int32_t ticket);
/* Tester_FRCNN:testOne with its test-time options (Tester_FRCNN.lua:54-139) in one stream-ordered pass, nothing but the
 * inputs and the final results crossing the bus: pass 1 = detect on the proposals, clamped to the image (:72-78); passes
 * 2..num_iter = detect on nn.SelectBoxes of the previous pass (:82-89; cached trunk features, not clamped, as the
 * reference); use_rbox_scores: the scores of pass i + 1 with the boxes of pass i (:91-97); the joined rows (:99-100,
 * n_out = R * (num_iter - use_rbox_scores)) are gathered per class with score > score_thresh and NMS'ed (:106-117);
 * bbox_voting: utils.bbox_vote of every kept box over its class's gathered rows, scores raised to vote_score_pow
 * (:118-124; 1 = untouched; other powers use the device powf, not libm's).
 * Outputs (host, synchronous; any may be NULL): scores n_out x C, bboxes n_out x 4C (the joined raw outputs :138),
 * keep_idx (C-1) x n_out rows into them in emission order, keep_counts C-1, voted (C-1) x n_out x 5 (row i of class j =
 * the voted box of keep_idx[j][i]; required when bbox_voting).                                                      */
typedef struct mpn_test_opts {
  int32_t num_iter;          /* opt.test_num_iterative_loc (>= 1) */
  int32_t use_rbox_scores;   /* opt.test_use_rbox_scores */
  int32_t bbox_voting;       /* opt.test_bbox_voting */
  float score_thresh;        /* Tester.thresh (-1.5, Tester_FRCNN.lua:50) */
  float nms_thr;             /* opt.test_nms_threshold (0.3) */
  float vote_thr;            /* opt.test_bbox_voting_nms_threshold (0.5) */
  float vote_score_pow;      /* opt.test_bbox_voting_score_pow (1) */
} mpn_test_opts;
int mpn_model_test_one(mpn_model *m, const float *image, int32_t H, int32_t W, const float *boxes, int64_t R,
                       float im_scale, float W0, float H0, const mpn_test_opts *opts, float *scores, float *bboxes,
                       int32_t *keep_idx, int32_t *keep_counts, float *voted);
/* Same with every buffer resident on the device, fully asynchronous (the
 * throughput path: bench.py `value`). */
int mpn_model_detect_nms_dev(mpn_model *m, const float *image_dev, int32_t H, int32_t W,
                             const float *boxes_dev, int64_t R, float im_scale, float W0, float H0,
                             float score_thresh, float nms_thr, float *scores_dev,
                             float *bboxes_dev, int32_t *keep_idx_dev, int32_t *keep_counts_dev);
/* mpn_model_detect_nms for N images in one stream-ordered pass: images N x 3 x H x W as mpn_model_trunk_batch. boxes:
 * R_total x 4, ORIGINAL coordinates of their own image; image i owns rows [img_offsets[i], img_offsets[i+1]) (host, N + 1
 * entries, img_offsets[0] = 0, every R_i >= 1, R_total <= max_rois). im_scale, W0, H0: host arrays of N. scores R_total x C,
 * bboxes R_total x 4C (clamped to their own image). keep_idx: image i's (C-1) x R_i block starts at (C-1) * img_offsets[i],
 * with row indices local to image i; keep_counts N x (C-1). Each image's slice is what mpn_model_detect_nms returns for that
 * image alone (the trunk's tensor-core plans depend on N, so its last bits may differ; entries of keep_idx past a class's
 * count are unspecified). With a detection sink set, N records are appended in image order. Any output may be NULL.
 * _dev: device buffers, stream-ordered; the host form is synchronous.                                                  */
int mpn_model_detect_nms_batch_dev(mpn_model *m, const float *images_dev, int32_t N, int32_t H, int32_t W,
                                   const float *boxes_dev, const int64_t *img_offsets, const float *im_scale,
                                   const float *W0, const float *H0, float score_thresh, float nms_thr,
                                   float *scores_dev, float *bboxes_dev, int32_t *keep_idx_dev, int32_t *keep_counts_dev);
int mpn_model_detect_nms_batch(mpn_model *m, const float *images, int32_t N, int32_t H, int32_t W,
                               const float *boxes, const int64_t *img_offsets, const float *im_scale,
                               const float *W0, const float *H0, float score_thresh, float nms_thr,
                               float *scores, float *bboxes, int32_t *keep_idx, int32_t *keep_counts);

/* ---- the detect tail after the network for a RANGE of classes (BASELINE configs[4], "NMS + BBoxNorm sweep": classes
 * shard across GPUs): nn.BBoxNorm (modules/BBoxNorm.lua:18-32; mean4 / std4 NULL = none) + utils.convertFrom per class
 * block (utils.lua:226-246) + clamp to [1,W0] x [1,H0] (Tester_FRCNN.lua:75-78) of deltas R x 4C against boxes R x 4
 * -> bboxes R x 4C, then for the foreground classes c in [c_begin, c_end) (1 <= c < C): rows with scores[:, c] >
 * score_thresh gathered and NMS'ed (Tester_FRCNN.lua:106-117). keep_idx (c_end - c_begin) x R proposal rows in emission
 * order, keep_counts c_end - c_begin. Device buffers, stream-ordered.                                              */
int mpn_post_detect_dev(mpn_ctx *ctx, const float *scores_dev, const float *deltas_dev, const float *boxes_dev, int64_t R,
                        int32_t C, const float *mean4, const float *std4, float W0, float H0, float score_thresh,
                        float nms_thr, int32_t c_begin, int32_t c_end, float *bboxes_dev, int32_t *keep_idx_dev,
                        int32_t *keep_counts_dev);

/* ---- after NMS, on the device (SURVEY 8f-2/3, 8e) --------------------------------------------------------------
 * Detection record of one image = the result of utils.keep_top_k (utils.lua:75-96; Tester:keepTopKPerImage,
 * Tester_FRCNN.lua:163-168, test_runner.lua:121) over the image's per-class NMS output, in a fixed size so that the
 * end-of-run all-gather needs no size exchange: MPN_REC_FLOATS floats = [count, MPN_MAX_DET x (x1,y1,x2,y2,score,class)],
 * class = 1-based foreground class (the index of the reference's per-class table), rows class-major and in NMS
 * emission order inside a class (= the reference's tables after keep_top_k), unused rows zero. keep_top_k keeps every
 * row with score >= the top_k-th largest score, so ties at the cut make count exceed top_k; count > MPN_MAX_DET means
 * the record overflowed (rows beyond MPN_MAX_DET are dropped; the host mirrors raise).                              */
enum { MPN_MAX_DET = 128, MPN_REC_FLOATS = 769, MPN_DIST_ID_BYTES = 128 };
/* scores R x C, bboxes R x 4C (detect outputs), keep_idx (C-1) x cap proposal rows in emission order, keep_counts C-1
 * (the outputs of mpn_model_detect_nms*, cap = R there). Device buffers, stream-ordered; host form synchronous.   */
int mpn_pack_detections_dev(mpn_ctx *ctx, const float *scores_dev, const float *bboxes_dev, int64_t R, int32_t C,
                            const int32_t *keep_idx_dev, const int32_t *keep_counts_dev, int64_t cap, int32_t top_k,
                            float *record_dev);
int mpn_pack_detections(mpn_ctx *ctx, const float *scores, const float *bboxes, int64_t R, int32_t C,
                        const int32_t *keep_idx, const int32_t *keep_counts, int64_t cap, int32_t top_k, float *record);
/* nn.SelectBoxes:updateOutput (modules/SelectBoxes.lua:26-56; Tester_FRCNN.lua:82-90): out[r] = the 4 box values of
 * the class with the largest score in row r (first maximum, background included), * std4 + mean4 when both are given
 * (NULL, NULL: the "dry run" of SelectBoxes.lua:46-47). classes R x C, ys R x 4C, out R x 4.                      */
int mpn_select_boxes(mpn_ctx *ctx, const float *classes, const float *ys, int64_t R, int32_t C, const float *mean4,
                     const float *std4, float *out);
int mpn_select_boxes_dev(mpn_ctx *ctx, const float *classes_dev, const float *ys_dev, int64_t R, int32_t C,
                         const float *mean4, const float *std4, float *out_dev);
/* From now on every mpn_model_detect_nms / _dev / _submit call also packs the image's record (top_k, normally 100)
 * into records_dev[n * MPN_REC_FLOATS], n = 0, 1, ... (stream-ordered, one extra launch per image); the call fails
 * once `capacity` records were written. records_dev = NULL switches the sink off; setting it resets the count.      */
int mpn_model_set_detection_sink(mpn_model *m, float *records_dev, int64_t capacity, int32_t top_k);
int mpn_model_detection_sink_count(const mpn_model *m, int64_t *n_records);

/* ---- the path's ONE collective (SURVEY 8e; test_runner.lua:96-103,121-122 joins the per-image results of all
 * replicas): an NCCL all-gather of the packed records, issued by the library on the ctx stream. One process (or
 * thread) per GPU: rank 0 calls mpn_dist_unique_id and hands the MPN_DIST_ID_BYTES bytes to every rank by whatever
 * channel the host has (torch.distributed / a file / threads' shared memory), then every rank calls mpn_dist_init
 * concurrently. NCCL is bound at run time (the libnccl.so.2 already in the process, else the system one); without
 * it these calls fail with a message and nothing else is affected. A ctx without a communicator is a world of 1.    */
int mpn_dist_unique_id(mpn_ctx *ctx, uint8_t *id);
int mpn_dist_init(mpn_ctx *ctx, const uint8_t *id, int32_t rank, int32_t world);
int mpn_dist_world(const mpn_ctx *ctx, int32_t *rank, int32_t *world);
/* recv = world x n_floats, rank-major; every rank contributes n_floats (its records, padded to the same count).
 * _dev: device buffers, stream-ordered (send may alias its own slot of recv). Host form: recv_host, synchronous.    */
int mpn_dist_all_gather_dev(mpn_ctx *ctx, const float *send_dev, int64_t n_floats, float *recv_dev);
int mpn_dist_all_gather(mpn_ctx *ctx, const float *send_dev, int64_t n_floats, float *recv_host);
int mpn_dist_destroy(mpn_ctx *ctx);
int mpn_dist_nccl_version(mpn_ctx *ctx, int32_t *version);

/* introspection for tests: rows [r0, r0 + n) of the pooled tensor the LAST heads / detect call fed to tower `tower` —
 * the output of the fused Foveal + ROI pooling (+ per-level L2 normalise x 1000) kernel on the product path — as fp32
 * n x (PH*PW) x Ctot (channels-last, levels concatenated along channels; value = hi + lo of the split planes).
 * out may be NULL to query *R_total / *bins / *Ctot only. Host buffer, synchronous.                                 */
int mpn_model_get_pooled(mpn_model *m, int32_t tower, int64_t r0, int64_t n, float *out, int64_t capacity,
                         int64_t *R_total, int32_t *bins, int32_t *Ctot);
/* introspection for tests/profiling: copy a trunk slot to host as N x C x H x W fp32 (N = images of the last trunk call) */
int mpn_model_get_trunk_slot(mpn_model *m, int32_t slot, float *out_nchw, int64_t capacity,
                             int32_t *C, int32_t *H, int32_t *W);
/* select conv/GEMM implementation: 0 = tcgen05 tensor-core path (default, product),
 * 1 = plain fp32 CUDA-core check kernel (debug/verification only, very slow),
 * 2 = tcgen05 path with the conv -> 2x2 max-pool epilogue fusion disabled, so every trunk slot is
 *     materialised (mpn_model_get_trunk_slot fails loudly for a slot the fusion elided). */
int mpn_model_set_conv_impl(mpn_model *m, int32_t impl);
/* algorithmic FLOPs of the last trunk / heads call (SURVEY 8d definition)    */
int mpn_model_last_flops(const mpn_model *m, double *trunk_flops, double *head_flops);

/* standalone GEMM check entry (tests): C[M,N] = A[M,K] * B[N,K]^T + bias, fp32 host
 * buffers, computed with the same split-bf16 tcgen05 kernel the model uses (impl 0), the CUDA-core fp32 check kernel
 * (impl 1), or the fp16-weight two-product kernels of fc6 / fc7 (impl 2; needs N >= 1024).  */
int mpn_gemm_check(mpn_ctx *ctx, const float *A, const float *B, const float *bias, int64_t M,
                   int64_t N, int64_t K, int32_t relu, int32_t impl, float *C);
/* engine microbenchmark (diagnostics, tools/engine_sweep.py): times `iters` back-to-back launches of the tcgen05 engine on
 * device-resident random operands, C[M,N] = A[M,K] * B[N,K]^T, returns the mean milliseconds per launch and the chosen
 * configuration (BN, CTA group, split-K). */
int mpn_gemm_bench(mpn_ctx *ctx, int64_t M, int64_t N, int64_t K, int32_t iters, double *ms_per_launch,
                   int32_t *bn, int32_t *cta_group, int32_t *splitk);
/* conv microbenchmark with pipeline-wait counters of CTA 0 (3x3 A-reuse kernel only; all zero otherwise):
 * dbg[0..2] producer {wait emptyA, wait emptyB, total}, [3..6] MMA issuer {wait fullA, wait fullB, wait tempty, total},
 * [7..9] epilogue warp {wait tfull, store time, total} — SM cycles summed over the launch.
 * *mode: bit 0 = 3x3 A-reuse kernel, bit 4 = stream-K schedule. */
int mpn_conv_bench(mpn_ctx *ctx, int64_t N, int64_t Cin, int64_t H, int64_t W, int64_t Cout, int32_t k, int32_t stride,
                   int32_t pad, int32_t iters, double *ms_per_launch, int32_t *bn, int32_t *cta_group, int32_t *mode,
                   uint64_t *dbg16);
/* host-only view of the tcgen05 kernels' work walk (no GPU): the (tile, s0, s1) pieces scheduling unit `unit` of
 * `num_units` visits, in order, for `total_tiles` tiles of `steps_per_tile` K steps; streamk = 0: whole tiles round-robin,
 * 1: contiguous (tile, step) ranges in rotated order (continuation piece, head piece, whole tiles). pieces: max_pieces x 3. */
int mpn_debug_segwalk(int32_t streamk, int32_t unit, int32_t num_units, int32_t total_tiles, int32_t steps_per_tile,
                      int32_t *pieces, int32_t max_pieces, int32_t *n_pieces);
/* host-only view of the planner (no GPU): the engine configuration chosen for a conv / Linear layer (Cin multiple of 64) on
 * a device with sm_count SMs; per_roi = 1 for per-ROI layers (rounding-relevant choices from (Cout, K) only).
 * out[8] = {mode (bit 0: 3x3 A-reuse kernel), CTA group, N tile, split-K, stream-K, patch tn, th, tw}. */
int mpn_debug_plan(int64_t N, int64_t Cin, int64_t H, int64_t W, int64_t Cout, int32_t k, int32_t stride, int32_t pad,
                   int32_t per_roi, int32_t sm_count, int32_t *out);
/* standalone conv check entry (tests): x N x Cin x H x W, w Cout x Cin x kh x kw (Torch layouts) */
int mpn_conv_check(mpn_ctx *ctx, const float *x, int64_t N, int64_t Cin, int64_t H, int64_t W,
                   const float *w, const float *bias, int64_t Cout, int32_t kh, int32_t kw,
                   int32_t stride, int32_t pad, int32_t relu, int32_t impl, float *y);

/* MPN_CDEF_END */
#ifdef __cplusplus
}
#endif
#endif /* MPN_ABI_H */
