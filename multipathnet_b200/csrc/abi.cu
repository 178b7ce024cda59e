// abi.cu — context management and the host-buffer entry points of include/mpn_abi.h.
// Host-pointer calls stage through ctx-owned device scratch, run on the ctx stream and
// synchronise before returning (the reference's :cuda()/:float() copies block the same way).
#include "conv_gemm.cuh"
#include "roi.cuh"
#include <algorithm>
#include <mutex>

int mpn_nms_launch(mpn_ctx *, const float *, int, int, const int32_t *, const int32_t *, float, int32_t *, int32_t *);
int mpn_nms_dense_launch(mpn_ctx *, const float *, int, float, int32_t *, int32_t *);
int mpn_bbox_vote_launch(mpn_ctx *, const float *, int, const float *, int, float, float *);
int mpn_pack_detections_launch(mpn_ctx *, const float *, const float *, int, const int32_t *, const int32_t *, int, int, float *);
int mpn_gather_scored_range_launch(mpn_ctx *, const float *, const float *, int, int, int, int, float, float *, int32_t *, int32_t *);
int mpn_bbox_norm_decode_launch(mpn_ctx *, const float *, const float *, int64_t, int, int, float, float, float *, const float *, const float *);
int mpn_select_boxes_launch(mpn_ctx *, const float *, const float *, int64_t, int, const float *, const float *, float *);
int mpn_foveal_launch(mpn_ctx *, const float *, int64_t, float *);
int mpn_context_region_launch(mpn_ctx *, const float *, int64_t, float, float *);
int mpn_get_images_launch(mpn_ctx *, const float *, int32_t, int32_t, const mpn_image_transform *, int32_t, int32_t, float *);
int mpn_get_images_size_impl(int32_t, int32_t, double, double, int32_t *, int32_t *, double *);
int mpn_get_images_u8_launch(mpn_ctx *, const uint8_t *, int32_t, int32_t, const mpn_image_transform *, int32_t, int32_t, float *);
int mpn_get_images_batch_size_impl(int32_t, const int32_t *, const int32_t *, double, double, int32_t *, int32_t *, double *, int32_t *,
                                   int32_t *);
int mpn_get_images_batch_launch(mpn_ctx *, const float *, const uint8_t *, int32_t, const int32_t *, const int32_t *, const int32_t *,
                                const int32_t *, int32_t, int32_t, const mpn_image_transform *, float *);
int mpn_get_images_batch_check(mpn_ctx *, int32_t, const int32_t *, const int32_t *, const mpn_image_transform *, double, double, int32_t *,
                               int32_t *, double *, int32_t &, int32_t &, size_t &);
int mpn_bbox_norm_launch(mpn_ctx *, float *, int64_t, int64_t, const float *, const float *);
int mpn_bbox_decode_launch(mpn_ctx *, const float *, const float *, int64_t, int, int, float, float, float *);
int mpn_split_rows_launch(mpn_ctx *, const float *, int64_t, int64_t, int64_t, __nv_bfloat16 *, __nv_bfloat16 *, int64_t);
int mpn_nchw_to_nhwc_split_launch(mpn_ctx *, const float *, int, int, int, int, DTensor &);
int mpn_nhwc_split_to_nchw_launch(mpn_ctx *, const DTensor &, float *);
int mpn_weight_permute_split_launch(mpn_ctx *, const float *, int64_t, int, int, int, __nv_bfloat16 *, __nv_bfloat16 *);
int mpn_absmax(mpn_ctx *, const float *, int64_t, float *);
int mpn_weight_permute_half_launch(mpn_ctx *, const float *, int64_t, int, int, int, float, void *);
int mpn_split_rows_f16_launch(mpn_ctx *, const float *, int64_t, int64_t, int64_t, __nv_bfloat16 *, __nv_bfloat16 *, int64_t);

static std::string g_create_err;
static std::mutex g_create_mu;

static int grow(mpn_ctx *ctx, void **p, size_t *have, size_t bytes, void **out) {
  if (bytes > *have) {
    if (*p) { cudaStreamSynchronize(ctx->stream); cudaFree(*p); *p = nullptr; *have = 0; }
    size_t want = std::max(bytes, (size_t)1 << 20);
    MPN_CUDA(ctx, cudaMalloc(p, want));
    *have = want;
  }
  *out = *p;
  return MPN_OK;
}
int mpn_ovf_flag(mpn_ctx *ctx, unsigned **flag_dev) {
  if (!ctx->ovf_dev) {
    MPN_CUDA(ctx, cudaMalloc((void **)&ctx->ovf_dev, 256));
    MPN_CUDA(ctx, cudaMemsetAsync(ctx->ovf_dev, 0, 256, ctx->stream));
    MPN_CUDA(ctx, cudaHostAlloc((void **)&ctx->ovf_host, 64, cudaHostAllocDefault));
    *ctx->ovf_host = 0;
  }
  *flag_dev = ctx->ovf_dev;
  return MPN_OK;
}
int mpn_ovf_copy_async(mpn_ctx *ctx, cudaStream_t stream) {
  if (!ctx->ovf_dev) return MPN_OK;
  MPN_CUDA(ctx, cudaMemcpyAsync(ctx->ovf_host, ctx->ovf_dev, sizeof(unsigned), cudaMemcpyDeviceToHost, stream));
  return MPN_OK;
}
int mpn_ovf_test(mpn_ctx *ctx) {
  if (!ctx->ovf_dev || !*ctx->ovf_host) return MPN_OK;
  const unsigned bits = *ctx->ovf_host;
  *ctx->ovf_host = 0;
  MPN_CUDA(ctx, cudaMemsetAsync(ctx->ovf_dev, 0, sizeof(unsigned), ctx->stream));
  if (bits & MPN_FLAG_BAD_BATCH)
    return mpn_fail(ctx, MPN_ERR_ARG, "a ROI row's batch index (column 0, 1-based, ImageDetect.lua:69) lies outside [1, N] for the N "
                                      "images of the last trunk forward: results of this call are invalid");
  return mpn_fail(ctx, MPN_ERR_STATE, "an activation left fp16's range (|x| > 65504 or NaN) in the fp16-plane path of fc6 / fc7: results of this call are "
                                      "saturated; rerun with mpn_ctx_set_option(ctx, \"fc_w16\", 0) (or MPN_FC_W16=0) for the three-product bf16 path");
}
int mpn_scratch(mpn_ctx *ctx, size_t bytes, void **out) { return grow(ctx, &ctx->scratch, &ctx->scratch_bytes, bytes, out); }
int mpn_scratch2(mpn_ctx *ctx, size_t bytes, void **out) { return grow(ctx, &ctx->scratch2, &ctx->scratch2_bytes, bytes, out); }
int mpn_scratch3(mpn_ctx *ctx, size_t bytes, void **out) { return grow(ctx, &ctx->scratch3, &ctx->scratch3_bytes, bytes, out); }

// bump allocator over scratch slot 1 for the host-wrapper calls
struct Arena {
  mpn_ctx *ctx; size_t off = 0; char *base = nullptr; size_t cap = 0;
  std::vector<size_t> sizes;
  size_t reserve(size_t bytes) { size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; }
  int commit() { void *p; MPN_TRY(mpn_scratch(ctx, off + 256, &p)); base = (char *)p; cap = off; return MPN_OK; }
  template <class T> T *at(size_t o) { return reinterpret_cast<T *>(base + o); }
};

extern "C" {

const char *mpn_version(void) { return "mpn_b200 0.1 (sm_100a; tcgen05 bf16x3 engine)"; }

int mpn_ctx_create(int device, void *cuda_stream, mpn_ctx **out) {
  if (!out) return MPN_ERR_ARG;
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || device < 0 || device >= count) {
    std::lock_guard<std::mutex> lk(g_create_mu);
    g_create_err = e != cudaSuccess ? std::string("no CUDA device: ") + cudaGetErrorString(e)
                                    : "device ordinal out of range";
    cudaGetLastError();
    return MPN_ERR_CUDA;
  }
  cudaDeviceProp prop;
  e = cudaSetDevice(device);
  if (e == cudaSuccess) e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) {
    std::lock_guard<std::mutex> lk(g_create_mu);
    g_create_err = std::string("cudaSetDevice/GetDeviceProperties failed: ") + cudaGetErrorString(e);
    return MPN_ERR_CUDA;
  }
  if (prop.major != 10) {
    std::lock_guard<std::mutex> lk(g_create_mu);
    g_create_err = "libmpn_b200 is built for sm_100a (Blackwell B200) only; found sm_" + std::to_string(prop.major) +
                   std::to_string(prop.minor) + ". There is no fallback path.";
    return MPN_ERR_STATE;
  }
  mpn_ctx *c = new mpn_ctx();
  c->device = device; c->stream = (cudaStream_t)cuda_stream; c->sm_count = prop.multiProcessorCount;
  *out = c;
  return MPN_OK;
}

int mpn_ctx_create_stream(int device, int priority, mpn_ctx **out) {
  const int rc = mpn_ctx_create(device, nullptr, out);
  if (rc != MPN_OK) return rc;
  mpn_ctx *c = *out;
  int lo = 0, hi = 0;
  cudaDeviceGetStreamPriorityRange(&lo, &hi);                  // lo = numerically largest = least urgent
  const int pr = priority < hi ? hi : (priority > lo ? lo : priority);
  cudaStream_t s = nullptr;
  const cudaError_t e = cudaStreamCreateWithPriority(&s, cudaStreamNonBlocking, pr);
  if (e != cudaSuccess) {
    { std::lock_guard<std::mutex> lk(g_create_mu); g_create_err = std::string("cudaStreamCreateWithPriority failed: ") + cudaGetErrorString(e); }
    delete c; *out = nullptr;
    return MPN_ERR_CUDA;
  }
  c->stream = s; c->own_stream = 1;
  return MPN_OK;
}

void *mpn_ctx_stream(const mpn_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }

int mpn_ctx_wait_ctx(mpn_ctx *ctx, mpn_ctx *other) {
  if (!ctx || !other) return MPN_ERR_ARG;
  MPN_CHECK_ARG(ctx, ctx->device == other->device, "mpn_ctx_wait_ctx: both contexts must be on the same device");
  if (ctx == other || ctx->stream == other->stream) return MPN_OK;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  if (!ctx->join_ev) MPN_CUDA(ctx, cudaEventCreateWithFlags(&ctx->join_ev, cudaEventDisableTiming));
  MPN_CUDA(ctx, cudaEventRecord(ctx->join_ev, other->stream));
  MPN_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->join_ev, 0));
  return MPN_OK;
}

void mpn_ctx_destroy(mpn_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  mpn_dist_destroy(ctx);
  if (ctx->scratch) cudaFree(ctx->scratch);
  if (ctx->scratch2) cudaFree(ctx->scratch2);
  if (ctx->scratch3) cudaFree(ctx->scratch3);
  if (ctx->small_dev) cudaFree(ctx->small_dev);
  if (ctx->ovf_dev) cudaFree(ctx->ovf_dev);
  if (ctx->ovf_host) cudaFreeHost(ctx->ovf_host);
  if (ctx->u8_lut_dev) cudaFree(ctx->u8_lut_dev);
  if (ctx->sk_ws) cudaFree(ctx->sk_ws);
  if (ctx->sk_flags) cudaFree(ctx->sk_flags);
  if (ctx->tl_min) cudaFree(ctx->tl_min);
  if (ctx->tl_max) cudaFree(ctx->tl_max);
  for (auto &r : ctx->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  for (auto e : ctx->ev_pool) cudaEventDestroy(e);
  if (ctx->join_ev) cudaEventDestroy(ctx->join_ev);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char *mpn_last_error(const mpn_ctx *ctx) {
  if (!ctx) return g_create_err.c_str();
  return ctx->err.c_str();
}

int mpn_ctx_synchronize(mpn_ctx *ctx) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_TRY(mpn_ovf_copy_async(ctx, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return mpn_ovf_test(ctx);
}

int64_t mpn_ctx_launch_count(const mpn_ctx *ctx) { return ctx ? ctx->launches : -1; }

int mpn_ctx_set_option(mpn_ctx *ctx, const char *name, int64_t value) {
  if (!ctx || !name) return MPN_ERR_ARG;
  if (!strcmp(name, "roi_norm_split")) { ctx->opt_roi_norm_split = value < 0 ? -1 : (value ? 1 : 0); return MPN_OK; }
  if (!strcmp(name, "fc_w16")) { ctx->opt_fc_w16 = value < 0 ? -1 : (value ? 1 : 0); return MPN_OK; }
  if (!strcmp(name, "roi_impl")) {
    MPN_CHECK_ARG(ctx, value <= 5, "roi_impl: 0 = cluster kernel (st.async exchange), 1 = legacy staged, 2 = legacy two-pass, 3 = cluster kernel (barrier exchange), 4 = bulk-copy kernel, 5 = persistent ring kernel");
    ctx->opt_roi_impl = value < 0 ? -1 : (int)value; return MPN_OK;
  }
  return mpn_fail(ctx, MPN_ERR_ARG, std::string("unknown option: ") + name);
}

int mpn_ctx_timeline_begin(mpn_ctx *ctx, int32_t max_launches) {
  if (!ctx || max_launches <= 0) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  if (max_launches > ctx->tl_cap) {
    if (ctx->tl_min) { cudaFree(ctx->tl_min); cudaFree(ctx->tl_max); ctx->tl_min = ctx->tl_max = nullptr; }
    MPN_CUDA(ctx, cudaMalloc((void **)&ctx->tl_min, sizeof(unsigned long long) * 4 * (size_t)max_launches));
    MPN_CUDA(ctx, cudaMalloc((void **)&ctx->tl_max, sizeof(unsigned long long) * 4 * (size_t)max_launches));
    ctx->tl_cap = max_launches;
  }
  MPN_CUDA(ctx, cudaMemsetAsync(ctx->tl_min, 0xff, sizeof(unsigned long long) * 4 * (size_t)ctx->tl_cap, ctx->stream));
  MPN_CUDA(ctx, cudaMemsetAsync(ctx->tl_max, 0, sizeof(unsigned long long) * 4 * (size_t)ctx->tl_cap, ctx->stream));
  ctx->tl_n = 0; ctx->tl_on = 1;
  return MPN_OK;
}

int mpn_ctx_timeline_end(mpn_ctx *ctx, uint64_t *stamps_min, uint64_t *stamps_max, int32_t *n_launches) {
  if (!ctx || !stamps_min || !stamps_max || !n_launches) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  ctx->tl_on = 0;
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  const int n = std::min(ctx->tl_n, ctx->tl_cap);
  MPN_CUDA(ctx, cudaMemcpy(stamps_min, ctx->tl_min, sizeof(uint64_t) * 4 * (size_t)n, cudaMemcpyDeviceToHost));
  MPN_CUDA(ctx, cudaMemcpy(stamps_max, ctx->tl_max, sizeof(uint64_t) * 4 * (size_t)n, cudaMemcpyDeviceToHost));
  *n_launches = n;
  return MPN_OK;
}

int mpn_ctx_profile_begin(mpn_ctx *ctx) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  for (auto &r : ctx->prof) { ctx->ev_pool.push_back(r.a); ctx->ev_pool.push_back(r.b); }
  ctx->prof.clear();
  ctx->profiling = 1;
  return MPN_OK;
}

int mpn_ctx_profile_end(mpn_ctx *ctx, double *ms_by_cat, int64_t *launches_by_cat) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  ctx->profiling = 0;
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int c = 0; c < MPN_NCAT; ++c) { if (ms_by_cat) ms_by_cat[c] = 0.0; if (launches_by_cat) launches_by_cat[c] = 0; }
  for (auto &r : ctx->prof) {
    float ms = 0.f;
    MPN_CUDA(ctx, cudaEventElapsedTime(&ms, r.a, r.b));
    if (ms_by_cat) ms_by_cat[r.cat] += ms;
    if (launches_by_cat) launches_by_cat[r.cat] += 1;
    ctx->ev_pool.push_back(r.a); ctx->ev_pool.push_back(r.b);
  }
  ctx->prof.clear();
  return MPN_OK;
}

// ------------------------------------------------------------------ NMS family
int mpn_nms_batched_dev(mpn_ctx *ctx, const float *scored_boxes_dev, const int64_t *seg_offsets, int64_t nseg,
                        float thr, int32_t *keep_idx_dev, int32_t *keep_counts_dev) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, seg_offsets && nseg >= 0, "seg_offsets missing");
  if (nseg == 0) return MPN_OK;
  // device form requires uniform segments (the pipeline's layout: nseg x cap x 5)
  const int64_t cap = seg_offsets[1] - seg_offsets[0];
  for (int64_t s = 0; s < nseg; ++s)
    MPN_CHECK_ARG(ctx, seg_offsets[s + 1] - seg_offsets[s] == cap && seg_offsets[s] == s * cap,
                  "mpn_nms_batched_dev needs uniform contiguous segments");
  if (cap == 0) { MPN_CUDA(ctx, cudaMemsetAsync(keep_counts_dev, 0, sizeof(int32_t) * nseg, ctx->stream)); return MPN_OK; }
  return mpn_nms_launch(ctx, scored_boxes_dev, (int)cap, (int)nseg, nullptr, nullptr, thr, keep_idx_dev, keep_counts_dev);
}

int mpn_nms_batched(mpn_ctx *ctx, const float *scored_boxes, const int64_t *seg_offsets, int64_t nseg, float thr,
                    int32_t *keep_idx, int64_t *keep_counts) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, seg_offsets && keep_counts && nseg >= 0, "bad arguments");
  if (nseg == 0) return MPN_OK;
  int64_t cap = 0;
  for (int64_t s = 0; s < nseg; ++s) {
    MPN_CHECK_ARG(ctx, seg_offsets[s + 1] >= seg_offsets[s], "seg_offsets must be non-decreasing");
    cap = std::max(cap, seg_offsets[s + 1] - seg_offsets[s]);
  }
  for (int64_t s = 0; s < nseg; ++s) keep_counts[s] = 0;
  if (cap == 0) return MPN_OK;
  MPN_CHECK_ARG(ctx, scored_boxes && keep_idx, "buffers missing");
  MPN_CHECK_ARG(ctx, cap <= 0x7fffffff / 8, "segment too large");
  // repack ragged segments into the uniform-capacity device layout
  std::vector<float> packed((size_t)nseg * cap * 5, 0.f);
  std::vector<int32_t> counts(nseg);
  for (int64_t s = 0; s < nseg; ++s) {
    const int64_t n = seg_offsets[s + 1] - seg_offsets[s];
    counts[s] = (int32_t)n;
    if (n) memcpy(&packed[(size_t)s * cap * 5], scored_boxes + seg_offsets[s] * 5, sizeof(float) * 5 * (size_t)n);
  }
  Arena a{ctx};
  size_t o_sb = a.reserve(sizeof(float) * packed.size()), o_cnt = a.reserve(sizeof(int32_t) * nseg),
         o_keep = a.reserve(sizeof(int32_t) * (size_t)nseg * cap), o_kc = a.reserve(sizeof(int32_t) * nseg);
  MPN_TRY(a.commit());
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o_sb), packed.data(), sizeof(float) * packed.size(), cudaMemcpyHostToDevice, ctx->stream));
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<int32_t>(o_cnt), counts.data(), sizeof(int32_t) * nseg, cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(mpn_nms_launch(ctx, a.at<float>(o_sb), (int)cap, (int)nseg, a.at<int32_t>(o_cnt), nullptr, thr,
                         a.at<int32_t>(o_keep), a.at<int32_t>(o_kc)));
  std::vector<int32_t> hk((size_t)nseg * cap), hc(nseg);
  MPN_CUDA(ctx, cudaMemcpyAsync(hk.data(), a.at<int32_t>(o_keep), sizeof(int32_t) * hk.size(), cudaMemcpyDeviceToHost, ctx->stream));
  MPN_CUDA(ctx, cudaMemcpyAsync(hc.data(), a.at<int32_t>(o_kc), sizeof(int32_t) * nseg, cudaMemcpyDeviceToHost, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int64_t s = 0; s < nseg; ++s) {
    keep_counts[s] = hc[s];
    if (hc[s]) memcpy(keep_idx + seg_offsets[s], &hk[(size_t)s * cap], sizeof(int32_t) * (size_t)hc[s]);
  }
  return MPN_OK;
}

int mpn_nms(mpn_ctx *ctx, const float *scored_boxes, int64_t N, float thr, int32_t *keep_idx, int64_t *n_keep) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CHECK_ARG(ctx, n_keep && N >= 0, "bad arguments");
  int64_t offs[2] = {0, N};
  return mpn_nms_batched(ctx, scored_boxes, offs, 1, thr, keep_idx, n_keep);
}

int mpn_nms_dense(mpn_ctx *ctx, const float *scored_boxes, int64_t N, float thr, int32_t *pick_idx, int64_t *n_pick) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, n_pick && N >= 0, "bad arguments");
  *n_pick = 0;
  if (N == 0) return MPN_OK;     // utils.lua:405-407 returns an empty LongTensor
  MPN_CHECK_ARG(ctx, scored_boxes && pick_idx, "buffers missing");
  Arena a{ctx};
  size_t o_sb = a.reserve(sizeof(float) * 5 * (size_t)N), o_pick = a.reserve(sizeof(int32_t) * (size_t)N), o_cnt = a.reserve(16);
  MPN_TRY(a.commit());
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o_sb), scored_boxes, sizeof(float) * 5 * (size_t)N, cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(mpn_nms_dense_launch(ctx, a.at<float>(o_sb), (int)N, thr, a.at<int32_t>(o_pick), a.at<int32_t>(o_cnt)));
  int32_t cnt = 0;
  MPN_CUDA(ctx, cudaMemcpyAsync(&cnt, a.at<int32_t>(o_cnt), sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (cnt) MPN_CUDA(ctx, cudaMemcpy(pick_idx, a.at<int32_t>(o_pick), sizeof(int32_t) * (size_t)cnt, cudaMemcpyDeviceToHost));
  *n_pick = cnt;
  return MPN_OK;
}

int mpn_bbox_vote(mpn_ctx *ctx, const float *nms_boxes, int64_t K, const float *scored_boxes, int64_t N, float thr,
                  float *res) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, K >= 0 && N >= 0, "bad arguments");
  if (K == 0) return MPN_OK;
  MPN_CHECK_ARG(ctx, nms_boxes && res && (N == 0 || scored_boxes), "buffers missing");
  Arena a{ctx};
  size_t o_n = a.reserve(sizeof(float) * 5 * (size_t)K), o_s = a.reserve(sizeof(float) * 5 * (size_t)std::max<int64_t>(N, 1)),
         o_r = a.reserve(sizeof(float) * 5 * (size_t)K);
  MPN_TRY(a.commit());
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o_n), nms_boxes, sizeof(float) * 5 * (size_t)K, cudaMemcpyHostToDevice, ctx->stream));
  if (N) MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o_s), scored_boxes, sizeof(float) * 5 * (size_t)N, cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(mpn_bbox_vote_launch(ctx, a.at<float>(o_n), (int)K, a.at<float>(o_s), (int)N, thr, a.at<float>(o_r)));
  MPN_CUDA(ctx, cudaMemcpyAsync(res, a.at<float>(o_r), sizeof(float) * 5 * (size_t)K, cudaMemcpyDeviceToHost, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MPN_OK;
}

// ------------------------------------------------------------------ the detect tail for a class range (BASELINE configs[4])
int mpn_post_detect_dev(mpn_ctx *ctx, const float *scores_dev, const float *deltas_dev, const float *boxes_dev, int64_t R, int32_t C,
                        const float *mean4, const float *std4, float W0, float H0, float score_thresh, float nms_thr, int32_t c_begin,
                        int32_t c_end, float *bboxes_dev, int32_t *keep_idx_dev, int32_t *keep_counts_dev) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, scores_dev && deltas_dev && boxes_dev && bboxes_dev && keep_idx_dev && keep_counts_dev && R > 0 && C >= 2, "buffers missing");
  MPN_CHECK_ARG(ctx, c_begin >= 1 && c_end <= C && c_begin < c_end, "class range must lie in [1, C)");
  MPN_CHECK_ARG(ctx, (mean4 == nullptr) == (std4 == nullptr), "mean4 and std4 go together");
  MPN_CHECK_ARG(ctx, R < (1ll << 31), "too many boxes");
  const int nseg = c_end - c_begin;
  // BBoxNorm + convertFrom + clamp of every class block (the decode is class-independent work: a rank that owns a class
  // range still decodes all of it only once per call; bytes are negligible next to the NMS)
  MPN_TRY(mpn_bbox_norm_decode_launch(ctx, deltas_dev, boxes_dev, R, C, 1, W0, H0, bboxes_dev, mean4, std4));
  // gather + NMS workspaces for this class range: scratch slot 1
  Arena a{ctx};
  size_t o_sb = a.reserve(sizeof(float) * 5 * (size_t)nseg * R), o_src = a.reserve(sizeof(int32_t) * (size_t)nseg * R),
         o_cnt = a.reserve(sizeof(int32_t) * (size_t)nseg);
  MPN_TRY(a.commit());
  MPN_TRY(mpn_gather_scored_range_launch(ctx, scores_dev, bboxes_dev, (int)R, C, c_begin, nseg, score_thresh, a.at<float>(o_sb),
                                         a.at<int32_t>(o_src), a.at<int32_t>(o_cnt)));
  return mpn_nms_launch(ctx, a.at<float>(o_sb), (int)R, nseg, a.at<int32_t>(o_cnt), a.at<int32_t>(o_src), nms_thr, keep_idx_dev, keep_counts_dev);
}

// ------------------------------------------------------------------ after NMS (post.cu)
int mpn_pack_detections_dev(mpn_ctx *ctx, const float *scores_dev, const float *bboxes_dev, int64_t R, int32_t C,
                            const int32_t *keep_idx_dev, const int32_t *keep_counts_dev, int64_t cap, int32_t top_k, float *record_dev) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, scores_dev && bboxes_dev && keep_idx_dev && keep_counts_dev && record_dev && R > 0 && cap > 0, "buffers missing");
  return mpn_pack_detections_launch(ctx, scores_dev, bboxes_dev, C, keep_idx_dev, keep_counts_dev, (int)cap, top_k, record_dev);
}

int mpn_pack_detections(mpn_ctx *ctx, const float *scores, const float *bboxes, int64_t R, int32_t C, const int32_t *keep_idx,
                        const int32_t *keep_counts, int64_t cap, int32_t top_k, float *record) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, scores && bboxes && keep_idx && keep_counts && record && R > 0 && C >= 2 && cap > 0, "buffers missing");
  Arena a{ctx};
  const size_t bs = sizeof(float) * (size_t)R * C, bb = sizeof(float) * (size_t)R * 4 * C, bk = sizeof(int32_t) * (size_t)(C - 1) * cap,
               bc = sizeof(int32_t) * (size_t)(C - 1), br = sizeof(float) * MPN_REC_FLOATS;
  size_t o_s = a.reserve(bs), o_b = a.reserve(bb), o_k = a.reserve(bk), o_c = a.reserve(bc), o_r = a.reserve(br);
  MPN_TRY(a.commit());
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o_s), scores, bs, cudaMemcpyHostToDevice, ctx->stream));
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o_b), bboxes, bb, cudaMemcpyHostToDevice, ctx->stream));
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<int32_t>(o_k), keep_idx, bk, cudaMemcpyHostToDevice, ctx->stream));
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<int32_t>(o_c), keep_counts, bc, cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(mpn_pack_detections_launch(ctx, a.at<float>(o_s), a.at<float>(o_b), C, a.at<int32_t>(o_k), a.at<int32_t>(o_c), (int)cap, top_k,
                                     a.at<float>(o_r)));
  MPN_CUDA(ctx, cudaMemcpyAsync(record, a.at<float>(o_r), br, cudaMemcpyDeviceToHost, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MPN_OK;
}

int mpn_select_boxes_dev(mpn_ctx *ctx, const float *classes_dev, const float *ys_dev, int64_t R, int32_t C, const float *mean4,
                         const float *std4, float *out_dev) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, R >= 0 && C >= 1 && (R == 0 || (classes_dev && ys_dev && out_dev)), "buffers missing");
  MPN_CHECK_ARG(ctx, (mean4 == nullptr) == (std4 == nullptr), "mean4 and std4 go together");
  return mpn_select_boxes_launch(ctx, classes_dev, ys_dev, R, C, mean4, std4, out_dev);
}

int mpn_select_boxes(mpn_ctx *ctx, const float *classes, const float *ys, int64_t R, int32_t C, const float *mean4, const float *std4,
                     float *out) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, R >= 0 && C >= 1, "bad arguments");
  if (R == 0) return MPN_OK;
  MPN_CHECK_ARG(ctx, classes && ys && out, "buffers missing");
  Arena a{ctx};
  const size_t bs = sizeof(float) * (size_t)R * C, bb = sizeof(float) * (size_t)R * 4 * C, bo = sizeof(float) * (size_t)R * 4;
  size_t o_s = a.reserve(bs), o_b = a.reserve(bb), o_o = a.reserve(bo);
  MPN_TRY(a.commit());
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o_s), classes, bs, cudaMemcpyHostToDevice, ctx->stream));
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o_b), ys, bb, cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(mpn_select_boxes_dev(ctx, a.at<float>(o_s), a.at<float>(o_b), R, C, mean4, std4, a.at<float>(o_o)));
  MPN_CUDA(ctx, cudaMemcpyAsync(out, a.at<float>(o_o), bo, cudaMemcpyDeviceToHost, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MPN_OK;
}

// ------------------------------------------------------------------ region modules
static int unary_rois(mpn_ctx *ctx, const float *in, int64_t R, int64_t out_rows_per_in, float *out,
                      int (*launch)(mpn_ctx *, const float *, int64_t, float, float *), float param) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, R >= 0, "bad R");
  if (R == 0) return MPN_OK;
  MPN_CHECK_ARG(ctx, in && out, "buffers missing");
  Arena a{ctx};
  size_t o_i = a.reserve(sizeof(float) * 5 * (size_t)R), o_o = a.reserve(sizeof(float) * 5 * (size_t)(R * out_rows_per_in));
  MPN_TRY(a.commit());
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o_i), in, sizeof(float) * 5 * (size_t)R, cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(launch(ctx, a.at<float>(o_i), R, param, a.at<float>(o_o)));
  MPN_CUDA(ctx, cudaMemcpyAsync(out, a.at<float>(o_o), sizeof(float) * 5 * (size_t)(R * out_rows_per_in), cudaMemcpyDeviceToHost, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MPN_OK;
}
static int foveal_adapter(mpn_ctx *c, const float *i, int64_t R, float, float *o) { return mpn_foveal_launch(c, i, R, o); }

int mpn_foveal(mpn_ctx *ctx, const float *rois, int64_t R, float *out) { return unary_rois(ctx, rois, R, 4, out, foveal_adapter, 0.f); }
int mpn_context_region(mpn_ctx *ctx, const float *rois, int64_t R, float scale, float *out) {
  return unary_rois(ctx, rois, R, 1, out, mpn_context_region_launch, scale);
}

// device-resident variants (stream-ordered, no copies): what a CudaTensor nn.Module forwards through — the reference's
// Foveal moves its input to the host and back (Foveal.lua:21-22,42); these do not
int mpn_foveal_dev(mpn_ctx *ctx, const float *rois_dev, int64_t R, float *out_dev) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, R >= 0, "bad R");
  if (R == 0) return MPN_OK;
  MPN_CHECK_ARG(ctx, rois_dev && out_dev, "buffers missing");
  return mpn_foveal_launch(ctx, rois_dev, R, out_dev);
}
int mpn_context_region_dev(mpn_ctx *ctx, const float *rois_dev, int64_t R, float scale, float *out_dev) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, R >= 0, "bad R");
  if (R == 0) return MPN_OK;
  MPN_CHECK_ARG(ctx, rois_dev && out_dev, "buffers missing");
  return mpn_context_region_launch(ctx, rois_dev, R, scale, out_dev);
}
int mpn_bbox_norm_dev(mpn_ctx *ctx, float *deltas_dev, int64_t R, int64_t C4, const float *mean4, const float *std4) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, R >= 0 && C4 > 0 && C4 % 4 == 0, "BBoxNorm: input:size(2) % 4 == 0 required (BBoxNorm.lua:19)");
  if (R == 0) return MPN_OK;
  MPN_CHECK_ARG(ctx, deltas_dev && mean4 && std4, "buffers missing");
  return mpn_bbox_norm_launch(ctx, deltas_dev, R, C4, mean4, std4);        // mean4 / std4 are HOST pointers (4 floats each)
}

// ------------------------------------------------------------------ getImages (SURVEY 8f-1)
int mpn_get_images_size(int32_t H0, int32_t W0, double scale, double max_size, int32_t *h, int32_t *w, double *im_scale) {
  return mpn_get_images_size_impl(H0, W0, scale, max_size, h, w, im_scale);
}
int mpn_get_images_dev(mpn_ctx *ctx, const float *im_dev, int32_t H0, int32_t W0, const mpn_image_transform *tf,
                       int32_t h, int32_t w, float *out_dev) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  return mpn_get_images_launch(ctx, im_dev, H0, W0, tf, h, w, out_dev);
}
int mpn_get_images_u8_dev(mpn_ctx *ctx, const uint8_t *im_hwc_dev, int32_t H0, int32_t W0, const mpn_image_transform *tf,
                          int32_t h, int32_t w, float *out_dev) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  return mpn_get_images_u8_launch(ctx, im_hwc_dev, H0, W0, tf, h, w, out_dev);
}
int mpn_get_images_u8(mpn_ctx *ctx, const uint8_t *im_hwc, int32_t H0, int32_t W0, const mpn_image_transform *tf,
                      int32_t h, int32_t w, float *out) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, im_hwc && out && tf && H0 > 0 && W0 > 0 && h > 0 && w > 0, "getImages: buffers missing or bad sizes");
  Arena a{ctx};
  const size_t bi = (size_t)H0 * W0 * 3, bo = sizeof(float) * 3 * (size_t)h * w;
  size_t o_i = a.reserve(bi), o_o = a.reserve(bo);
  MPN_TRY(a.commit());
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<uint8_t>(o_i), im_hwc, bi, cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(mpn_get_images_u8_launch(ctx, a.at<uint8_t>(o_i), H0, W0, tf, h, w, a.at<float>(o_o)));
  MPN_CUDA(ctx, cudaMemcpyAsync(out, a.at<float>(o_o), bo, cudaMemcpyDeviceToHost, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MPN_OK;
}
int mpn_get_images_batch_size(int32_t N, const int32_t *H0, const int32_t *W0, double scale, double max_size, int32_t *h, int32_t *w,
                              double *im_scale, int32_t *H, int32_t *W) {
  return mpn_get_images_batch_size_impl(N, H0, W0, scale, max_size, h, w, im_scale, H, W);
}
int mpn_get_images_batch_u8_dev(mpn_ctx *ctx, const uint8_t *ims_hwc_dev, int32_t N, const int32_t *H0, const int32_t *W0,
                                const mpn_image_transform *tf, double scale, double max_size, float *out_dev) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, ims_hwc_dev && out_dev, "getImages: buffers missing");
  int32_t h[MPN_MAX_BATCH], w[MPN_MAX_BATCH], H = 0, W = 0; size_t bi = 0;
  MPN_TRY(mpn_get_images_batch_check(ctx, N, H0, W0, tf, scale, max_size, h, w, nullptr, H, W, bi));
  return mpn_get_images_batch_launch(ctx, nullptr, ims_hwc_dev, N, H0, W0, h, w, H, W, tf, out_dev);
}
int mpn_get_images_batch_u8(mpn_ctx *ctx, const uint8_t *ims_hwc, int32_t N, const int32_t *H0, const int32_t *W0,
                            const mpn_image_transform *tf, double scale, double max_size, float *out) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, ims_hwc && out, "getImages: buffers missing");
  int32_t h[MPN_MAX_BATCH], w[MPN_MAX_BATCH], H = 0, W = 0; size_t bi = 0;
  MPN_TRY(mpn_get_images_batch_check(ctx, N, H0, W0, tf, scale, max_size, h, w, nullptr, H, W, bi));
  Arena a{ctx};
  const size_t bo = sizeof(float) * 3 * (size_t)N * H * W;
  size_t o_i = a.reserve(bi), o_o = a.reserve(bo);
  MPN_TRY(a.commit());
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<uint8_t>(o_i), ims_hwc, bi, cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(mpn_get_images_batch_launch(ctx, nullptr, a.at<uint8_t>(o_i), N, H0, W0, h, w, H, W, tf, a.at<float>(o_o)));
  MPN_CUDA(ctx, cudaMemcpyAsync(out, a.at<float>(o_o), bo, cudaMemcpyDeviceToHost, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MPN_OK;
}
int mpn_get_images(mpn_ctx *ctx, const float *im, int32_t H0, int32_t W0, const mpn_image_transform *tf,
                   int32_t h, int32_t w, float *out) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, im && out && tf && H0 > 0 && W0 > 0 && h > 0 && w > 0, "getImages: buffers missing or bad sizes");
  Arena a{ctx};
  const size_t bi = sizeof(float) * 3 * (size_t)H0 * W0, bo = sizeof(float) * 3 * (size_t)h * w;
  size_t o_i = a.reserve(bi), o_o = a.reserve(bo);
  MPN_TRY(a.commit());
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o_i), im, bi, cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(mpn_get_images_launch(ctx, a.at<float>(o_i), H0, W0, tf, h, w, a.at<float>(o_o)));
  MPN_CUDA(ctx, cudaMemcpyAsync(out, a.at<float>(o_o), bo, cudaMemcpyDeviceToHost, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MPN_OK;
}

int mpn_bbox_norm(mpn_ctx *ctx, float *deltas, int64_t R, int64_t C4, const float *mean4, const float *std4) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, R >= 0 && C4 > 0 && C4 % 4 == 0, "BBoxNorm: input:size(2) % 4 == 0 required (BBoxNorm.lua:19)");
  if (R == 0) return MPN_OK;
  MPN_CHECK_ARG(ctx, deltas && mean4 && std4, "buffers missing");
  Arena a{ctx};
  size_t o = a.reserve(sizeof(float) * (size_t)(R * C4));
  MPN_TRY(a.commit());
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o), deltas, sizeof(float) * (size_t)(R * C4), cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(mpn_bbox_norm_launch(ctx, a.at<float>(o), R, C4, mean4, std4));
  MPN_CUDA(ctx, cudaMemcpyAsync(deltas, a.at<float>(o), sizeof(float) * (size_t)(R * C4), cudaMemcpyDeviceToHost, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MPN_OK;
}

int mpn_bbox_decode(mpn_ctx *ctx, const float *deltas, const float *boxes, int64_t R, int64_t C, float *out) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, R >= 0 && C > 0, "bad arguments");
  if (R == 0) return MPN_OK;
  MPN_CHECK_ARG(ctx, deltas && boxes && out, "buffers missing");
  Arena a{ctx};
  size_t o_d = a.reserve(sizeof(float) * 4 * (size_t)(R * C)), o_b = a.reserve(sizeof(float) * 4 * (size_t)R),
         o_o = a.reserve(sizeof(float) * 4 * (size_t)(R * C));
  MPN_TRY(a.commit());
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o_d), deltas, sizeof(float) * 4 * (size_t)(R * C), cudaMemcpyHostToDevice, ctx->stream));
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o_b), boxes, sizeof(float) * 4 * (size_t)R, cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(mpn_bbox_decode_launch(ctx, a.at<float>(o_d), a.at<float>(o_b), R, (int)C, 0, 0.f, 0.f, a.at<float>(o_o)));
  MPN_CUDA(ctx, cudaMemcpyAsync(out, a.at<float>(o_o), sizeof(float) * 4 * (size_t)(R * C), cudaMemcpyDeviceToHost, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MPN_OK;
}

// ------------------------------------------------------------------ inn.ROIPooling
int mpn_roi_pool_dev(mpn_ctx *ctx, const float *fmap_dev, int64_t N, int64_t C, int64_t H, int64_t W,
                     const float *rois_dev, int64_t R, int32_t PW, int32_t PH, float spatial_scale, int32_t variant,
                     float *out_dev, int32_t *argmax_dev) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, N > 0 && C > 0 && H > 0 && W > 0 && R >= 0 && PW > 0 && PH > 0, "bad geometry");
  MPN_CHECK_ARG(ctx, variant == 1 || variant == 2, "variant must be 1 or 2");
  return mpn_roi_pool_nchw_launch(ctx, fmap_dev, N, C, H, W, rois_dev, R, PW, PH, spatial_scale, variant, out_dev, argmax_dev);
}

int mpn_roi_pool(mpn_ctx *ctx, const float *fmap, int64_t N, int64_t C, int64_t H, int64_t W, const float *rois,
                 int64_t R, int32_t PW, int32_t PH, float spatial_scale, int32_t variant, float *out, int32_t *argmax) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, N > 0 && C > 0 && H > 0 && W > 0 && R >= 0 && PW > 0 && PH > 0, "bad geometry");
  if (R == 0) return MPN_OK;
  MPN_CHECK_ARG(ctx, fmap && rois && out, "buffers missing");
  for (int64_t r = 0; r < R; ++r) {
    const float b = rois[5 * r];
    MPN_CHECK_ARG(ctx, b >= 1.f && b <= (float)N, "ROI batch index out of range (1-based, ImageDetect.lua:69)");
  }
  const size_t nf = (size_t)(N * C * H * W), no = (size_t)(R * C * PH * PW);
  Arena a{ctx};
  size_t o_f = a.reserve(sizeof(float) * nf), o_r = a.reserve(sizeof(float) * 5 * (size_t)R), o_o = a.reserve(sizeof(float) * no),
         o_a = a.reserve(sizeof(int32_t) * no);
  MPN_TRY(a.commit());
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o_f), fmap, sizeof(float) * nf, cudaMemcpyHostToDevice, ctx->stream));
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o_r), rois, sizeof(float) * 5 * (size_t)R, cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(mpn_roi_pool_dev(ctx, a.at<float>(o_f), N, C, H, W, a.at<float>(o_r), R, PW, PH, spatial_scale, variant,
                           a.at<float>(o_o), argmax ? a.at<int32_t>(o_a) : nullptr));
  MPN_CUDA(ctx, cudaMemcpyAsync(out, a.at<float>(o_o), sizeof(float) * no, cudaMemcpyDeviceToHost, ctx->stream));
  if (argmax) MPN_CUDA(ctx, cudaMemcpyAsync(argmax, a.at<int32_t>(o_a), sizeof(int32_t) * no, cudaMemcpyDeviceToHost, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MPN_OK;
}

// ------------------------------------------------------------------ engine check entries
int mpn_conv_check(mpn_ctx *ctx, const float *x, int64_t N, int64_t Cin, int64_t H, int64_t W, const float *w,
                   const float *bias, int64_t Cout, int32_t kh, int32_t kw, int32_t stride, int32_t pad, int32_t relu,
                   int32_t impl, float *y) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, x && w && y && N > 0 && Cin > 0 && Cout > 0 && H > 0 && W > 0, "bad arguments");
  const int64_t Ho = (H + 2 * pad - kh) / stride + 1, Wo = (W + 2 * pad - kw) / stride + 1;
  MPN_CHECK_ARG(ctx, Ho > 0 && Wo > 0, "empty output");
  const size_t nx = (size_t)(N * Cin * H * W), nw = (size_t)(Cout * Cin * kh * kw), ny = (size_t)(N * Cout * Ho * Wo);
  Arena a{ctx};
  size_t o_x = a.reserve(4 * nx), o_w = a.reserve(4 * nw), o_b = a.reserve(4 * (size_t)Cout), o_y = a.reserve(4 * ny),
         o_xh = a.reserve(2 * nx), o_xl = a.reserve(2 * nx), o_wh = a.reserve(2 * nw), o_wl = a.reserve(2 * nw),
         o_yh = a.reserve(2 * ny), o_yl = a.reserve(2 * ny);
  MPN_TRY(a.commit());
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o_x), x, 4 * nx, cudaMemcpyHostToDevice, ctx->stream));
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o_w), w, 4 * nw, cudaMemcpyHostToDevice, ctx->stream));
  if (bias) MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o_b), bias, 4 * (size_t)Cout, cudaMemcpyHostToDevice, ctx->stream));
  DTensor ty; ty.hi = a.at<__nv_bfloat16>(o_yh); ty.lo = a.at<__nv_bfloat16>(o_yl); ty.N = N; ty.H = Ho; ty.W = Wo; ty.C = Cout; ty.ld = Cout;
  if (impl == 2) {       // CUDA-core direct conv straight from the NCHW fp32 input (first-layer kernel)
    MPN_TRY(conv_direct_nchw_launch(ctx, a.at<float>(o_x), (int)N, (int)Cin, (int)H, (int)W, a.at<float>(o_w),
                                    bias ? a.at<float>(o_b) : nullptr, (int)Cout, kh, kw, stride, pad, relu, ty, w, bias));
  } else {
    DTensor tx; tx.hi = a.at<__nv_bfloat16>(o_xh); tx.lo = a.at<__nv_bfloat16>(o_xl); tx.N = N; tx.H = H; tx.W = W; tx.C = Cin; tx.ld = Cin;
    MPN_TRY(mpn_nchw_to_nhwc_split_launch(ctx, a.at<float>(o_x), (int)N, (int)Cin, (int)H, (int)W, tx));
    MPN_TRY(mpn_weight_permute_split_launch(ctx, a.at<float>(o_w), Cout, (int)Cin, kh, kw, a.at<__nv_bfloat16>(o_wh), a.at<__nv_bfloat16>(o_wl)));
    ConvProblem p; p.x = tx; p.w_hi = a.at<__nv_bfloat16>(o_wh); p.w_lo = a.at<__nv_bfloat16>(o_wl);
    p.bias = bias ? a.at<float>(o_b) : nullptr; p.Cout = (int)Cout; p.kh = kh; p.kw = kw; p.stride = stride; p.pad = pad; p.relu = relu;
    p.y = ty;
    if (impl == 1) { MPN_TRY(conv_ref_launch(ctx, p)); }
    else { ConvPlan pl; MPN_TRY(conv_tc_plan(ctx, p, pl)); MPN_TRY(conv_tc_launch(ctx, p, pl)); }
  }
  MPN_TRY(mpn_nhwc_split_to_nchw_launch(ctx, ty, a.at<float>(o_y)));
  MPN_CUDA(ctx, cudaMemcpyAsync(y, a.at<float>(o_y), 4 * ny, cudaMemcpyDeviceToHost, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MPN_OK;
}

int mpn_gemm_bench(mpn_ctx *ctx, int64_t M, int64_t N, int64_t K, int32_t iters, double *ms_per_launch, int32_t *bn,
                   int32_t *cta_group, int32_t *splitk) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, M > 0 && N > 0 && K > 0 && K % 64 == 0 && iters > 0 && ms_per_launch, "bad arguments");
  const size_t na = (size_t)(M * K), nb = (size_t)(N * K), nc = (size_t)(M * N);
  Arena a{ctx};
  size_t o_ah = a.reserve(2 * na), o_al = a.reserve(2 * na), o_bh = a.reserve(2 * nb), o_bl = a.reserve(2 * nb),
         o_ch = a.reserve(2 * nc + 64), o_cl = a.reserve(2 * nc + 64);
  MPN_TRY(a.commit());
  // operand contents do not matter for timing; 0x3c00-ish bf16 patterns keep everything finite
  MPN_CUDA(ctx, cudaMemsetAsync(a.at<char>(o_ah), 0x3c, 2 * na, ctx->stream));
  MPN_CUDA(ctx, cudaMemsetAsync(a.at<char>(o_al), 0x30, 2 * na, ctx->stream));
  MPN_CUDA(ctx, cudaMemsetAsync(a.at<char>(o_bh), 0x3c, 2 * nb, ctx->stream));
  MPN_CUDA(ctx, cudaMemsetAsync(a.at<char>(o_bl), 0x30, 2 * nb, ctx->stream));
  ConvProblem p;
  p.x.hi = a.at<__nv_bfloat16>(o_ah); p.x.lo = a.at<__nv_bfloat16>(o_al); p.x.N = M; p.x.H = 1; p.x.W = 1; p.x.C = K; p.x.ld = K;
  p.w_hi = a.at<__nv_bfloat16>(o_bh); p.w_lo = a.at<__nv_bfloat16>(o_bl); p.Cout = (int)N; p.relu = 1;
  const int64_t Npad = (N + 7) / 8 * 8;
  (void)Npad;
  if (N % 8 == 0) { p.y.hi = a.at<__nv_bfloat16>(o_ch); p.y.lo = a.at<__nv_bfloat16>(o_cl); }
  else { p.y.f32 = a.at<float>(o_ch); }
  p.y.N = M; p.y.H = 1; p.y.W = 1; p.y.C = N; p.y.ld = N; p.y_f32_ld = N;
  if (!(N % 8 == 0)) MPN_CHECK_ARG(ctx, 4 * nc <= 2 * (2 * nc + 64), "internal");
  ConvPlan pl;
  MPN_TRY(conv_tc_plan(ctx, p, pl));
  if (bn) *bn = pl.BN; if (cta_group) *cta_group = pl.CG; if (splitk) *splitk = pl.splitk;
  for (int i = 0; i < 3; ++i) MPN_TRY(conv_tc_launch(ctx, p, pl));
  cudaEvent_t e0, e1;
  MPN_CUDA(ctx, cudaEventCreate(&e0)); MPN_CUDA(ctx, cudaEventCreate(&e1));
  MPN_CUDA(ctx, cudaEventRecord(e0, ctx->stream));
  for (int i = 0; i < iters; ++i) MPN_TRY(conv_tc_launch(ctx, p, pl));
  MPN_CUDA(ctx, cudaEventRecord(e1, ctx->stream));
  MPN_CUDA(ctx, cudaEventSynchronize(e1));
  float ms = 0.f;
  MPN_CUDA(ctx, cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  *ms_per_launch = (double)ms / iters;
  return MPN_OK;
}

int mpn_conv_bench(mpn_ctx *ctx, int64_t N, int64_t Cin, int64_t H, int64_t W, int64_t Cout, int32_t k, int32_t stride,
                   int32_t pad, int32_t iters, double *ms_per_launch, int32_t *bn, int32_t *cta_group, int32_t *mode,
                   uint64_t *dbg16) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, N > 0 && Cin % 64 == 0 && Cout % 8 == 0 && iters > 0 && ms_per_launch, "bad arguments");
  const int64_t Ho = (H + 2 * pad - k) / stride + 1, Wo = (W + 2 * pad - k) / stride + 1;
  const size_t nx = (size_t)(N * H * W * Cin), nw = (size_t)(Cout * Cin * k * k), ny = (size_t)(N * Ho * Wo * Cout);
  Arena a{ctx};
  size_t o_xh = a.reserve(2 * nx), o_xl = a.reserve(2 * nx), o_wh = a.reserve(2 * nw), o_wl = a.reserve(2 * nw),
         o_yh = a.reserve(2 * ny), o_yl = a.reserve(2 * ny), o_dbg = a.reserve(16 * 8);
  MPN_TRY(a.commit());
  MPN_CUDA(ctx, cudaMemsetAsync(a.at<char>(o_xh), 0x3c, 2 * nx, ctx->stream));
  MPN_CUDA(ctx, cudaMemsetAsync(a.at<char>(o_xl), 0x30, 2 * nx, ctx->stream));
  MPN_CUDA(ctx, cudaMemsetAsync(a.at<char>(o_wh), 0x3c, 2 * nw, ctx->stream));
  MPN_CUDA(ctx, cudaMemsetAsync(a.at<char>(o_wl), 0x30, 2 * nw, ctx->stream));
  MPN_CUDA(ctx, cudaMemsetAsync(a.at<char>(o_dbg), 0, 128, ctx->stream));
  ConvProblem p;
  p.x.hi = a.at<__nv_bfloat16>(o_xh); p.x.lo = a.at<__nv_bfloat16>(o_xl); p.x.N = N; p.x.H = H; p.x.W = W; p.x.C = Cin; p.x.ld = Cin;
  p.w_hi = a.at<__nv_bfloat16>(o_wh); p.w_lo = a.at<__nv_bfloat16>(o_wl); p.Cout = (int)Cout; p.kh = k; p.kw = k; p.stride = stride; p.pad = pad; p.relu = 1;
  p.y.hi = a.at<__nv_bfloat16>(o_yh); p.y.lo = a.at<__nv_bfloat16>(o_yl); p.y.N = N; p.y.H = Ho; p.y.W = Wo; p.y.C = Cout; p.y.ld = Cout;
  ConvPlan pl;
  MPN_TRY(conv_tc_plan(ctx, p, pl));
  if (bn) *bn = pl.BN; if (cta_group) *cta_group = pl.CG; if (mode) *mode = pl.mode | (pl.streamk << 4);
  for (int i = 0; i < 3; ++i) MPN_TRY(conv_tc_launch(ctx, p, pl));
  cudaEvent_t e0, e1;
  MPN_CUDA(ctx, cudaEventCreate(&e0)); MPN_CUDA(ctx, cudaEventCreate(&e1));
  MPN_CUDA(ctx, cudaEventRecord(e0, ctx->stream));
  for (int i = 0; i < iters; ++i) MPN_TRY(conv_tc_launch(ctx, p, pl));
  MPN_CUDA(ctx, cudaEventRecord(e1, ctx->stream));
  MPN_CUDA(ctx, cudaEventSynchronize(e1));
  float ms = 0.f;
  MPN_CUDA(ctx, cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  *ms_per_launch = (double)ms / iters;
  if (dbg16) {       // one extra, instrumented launch
    p.dbg = a.at<char>(o_dbg);
    MPN_TRY(conv_tc_launch(ctx, p, pl));
    MPN_CUDA(ctx, cudaMemcpyAsync(dbg16, a.at<char>(o_dbg), 128, cudaMemcpyDeviceToHost, ctx->stream));
    MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return MPN_OK;
}

int mpn_gemm_check(mpn_ctx *ctx, const float *A, const float *B, const float *bias, int64_t M, int64_t N, int64_t K,
                   int32_t relu, int32_t impl, float *C) {
  if (!ctx) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, A && B && C && M > 0 && N > 0 && K > 0, "bad arguments");
  const size_t na = (size_t)(M * K), nb = (size_t)(N * K), nc = (size_t)(M * N);
  Arena a{ctx};
  size_t o_a = a.reserve(4 * na), o_b = a.reserve(4 * nb), o_bias = a.reserve(4 * (size_t)N), o_c = a.reserve(4 * nc),
         o_ah = a.reserve(2 * na), o_al = a.reserve(2 * na), o_bh = a.reserve(2 * nb), o_bl = a.reserve(2 * nb);
  MPN_TRY(a.commit());
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o_a), A, 4 * na, cudaMemcpyHostToDevice, ctx->stream));
  MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o_b), B, 4 * nb, cudaMemcpyHostToDevice, ctx->stream));
  if (bias) MPN_CUDA(ctx, cudaMemcpyAsync(a.at<float>(o_bias), bias, 4 * (size_t)N, cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(mpn_split_rows_launch(ctx, a.at<float>(o_a), M, K, K, a.at<__nv_bfloat16>(o_ah), a.at<__nv_bfloat16>(o_al), K));
  MPN_TRY(mpn_split_rows_launch(ctx, a.at<float>(o_b), N, K, K, a.at<__nv_bfloat16>(o_bh), a.at<__nv_bfloat16>(o_bl), K));
  ConvProblem p;
  p.x.hi = a.at<__nv_bfloat16>(o_ah); p.x.lo = a.at<__nv_bfloat16>(o_al); p.x.N = M; p.x.H = 1; p.x.W = 1; p.x.C = K; p.x.ld = K;
  p.w_hi = a.at<__nv_bfloat16>(o_bh); p.w_lo = a.at<__nv_bfloat16>(o_bl); p.bias = bias ? a.at<float>(o_bias) : nullptr;
  p.Cout = (int)N; p.relu = relu;
  p.m_invariant = 1;     // a Linear over independent rows: the result of a row must not depend on M
  p.y.f32 = a.at<float>(o_c); p.y.N = M; p.y.H = 1; p.y.W = 1; p.y.C = N; p.y.ld = N; p.y_f32_ld = N;
  if (impl == 1) { MPN_TRY(conv_ref_launch(ctx, p)); }
  else {
    if (impl == 2) {      // the fp16-weight ("w16") kernels: B as ONE fp16 plane of B * 2^e
      float amax = 0.f;
      MPN_TRY(mpn_absmax(ctx, a.at<float>(o_b), (int64_t)nb, &amax));
      int e = 0;
      if (amax > 0.f) { (void)frexpf(amax, &e); e = 14 - e; }
      const float sc = ldexpf(1.0f, e);
      MPN_TRY(mpn_weight_permute_half_launch(ctx, a.at<float>(o_b), N, (int)K, 1, 1, sc, a.at<void>(o_bh)));
      p.w16 = a.at<void>(o_bh); p.w16_inv_scale = 1.0f / sc; p.w_hi = p.w_lo = nullptr;
      MPN_TRY(mpn_split_rows_f16_launch(ctx, a.at<float>(o_a), M, K, K, a.at<__nv_bfloat16>(o_ah), a.at<__nv_bfloat16>(o_al), K));   // A as fp16 hi / lo planes
      p.x.fmt = 1;
    }
    ConvPlan pl; MPN_TRY(conv_tc_plan(ctx, p, pl)); MPN_TRY(conv_tc_launch(ctx, p, pl));
  }
  MPN_CUDA(ctx, cudaMemcpyAsync(C, a.at<float>(o_c), 4 * nc, cudaMemcpyDeviceToHost, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MPN_OK;
}

}  // extern "C"
