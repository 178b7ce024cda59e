// model.cu — executor for the detection graphs of models/{vgg,multipathnet,resnet}.lua,
// described as data (mpn_model_desc). Mirrors the reference's own trunk / heads split:
//   mpn_model_trunk  == model:get(1):forward            (ImageDetect.lua:107-108)
//   mpn_model_heads  == modules 2..n on cached features  (ImageDetect.lua:114-124)
//   mpn_model_detect == ImageDetect:detect tail          (ImageDetect.lua:176-192)
//   mpn_model_detect_nms adds Tester_FRCNN:testOne's clamp / per-class gather / NMS
//   (Tester_FRCNN.lua:75-78,106-117) so one stream-ordered pass produces final keep lists.
// All activations live in HBM as NHWC split-bf16 planes; every conv / Linear runs on the
// tcgen05 engine (gemm_tc.cu) except the Cin=3 first layer (conv_simt.cu).
#include "conv_gemm.cuh"
#include "roi.cuh"
#include <algorithm>
#include <cmath>
#include <map>
#include <memory>
#include <set>

// launchers defined in the other TUs
int mpn_maxpool_launch(mpn_ctx *, const DTensor &, int, int, int, DTensor &);
int mpn_avgpool_launch(mpn_ctx *, const DTensor &, DTensor &);
int mpn_weight_permute_split_launch(mpn_ctx *, const float *, int64_t, int, int, int, __nv_bfloat16 *, __nv_bfloat16 *);
int mpn_nhwc_split_to_nchw_launch(mpn_ctx *, const DTensor &, float *);
int mpn_project_rois_launch(mpn_ctx *, const float *, int64_t, float, float *);
int mpn_project_rois_batch_launch(mpn_ctx *, const float *, int64_t, const MpnBatch &, float *);
int mpn_detect_tail_batch_launch(mpn_ctx *, const float *, int64_t, int, int, int, float *, const float *, const float *, const MpnBatch &,
                                 float *, int, const float *, const float *);
int mpn_gather_scored_batch_launch(mpn_ctx *, const float *, const float *, int, float, const MpnBatch &, int, float *, int32_t *, int32_t *);
int mpn_get_images_launch(mpn_ctx *, const float *, int32_t, int32_t, const mpn_image_transform *, int32_t, int32_t, float *);
int mpn_get_images_size_impl(int32_t, int32_t, double, double, int32_t *, int32_t *, double *);
int mpn_get_images_u8_launch(mpn_ctx *, const uint8_t *, int32_t, int32_t, const mpn_image_transform *, int32_t, int32_t, float *);
int mpn_get_images_batch_launch(mpn_ctx *, const float *, const uint8_t *, int32_t, const int32_t *, const int32_t *, const int32_t *,
                                const int32_t *, int32_t, int32_t, const mpn_image_transform *, float *);
int mpn_get_images_batch_check(mpn_ctx *, int32_t, const int32_t *, const int32_t *, const mpn_image_transform *, double, double, int32_t *,
                               int32_t *, double *, int32_t &, int32_t &, size_t &);
int mpn_bbox_norm_launch(mpn_ctx *, float *, int64_t, int64_t, const float *, const float *);
int mpn_bbox_decode_launch(mpn_ctx *, const float *, const float *, int64_t, int, int, float, float, float *);
int mpn_softmax_mean_launch(mpn_ctx *, const float *, int64_t, int, int, int, float *);
int mpn_detect_tail_launch(mpn_ctx *, const float *, int64_t, int, int, int, float *, const float *, const float *, int, float, float,
                           float *, int, const float *, const float *);
int mpn_gather_scored_launch(mpn_ctx *, const float *, const float *, int, int, float, float *, int32_t *, int32_t *);
int mpn_nms_launch(mpn_ctx *, const float *, int, int, const int32_t *, const int32_t *, float, int32_t *, int32_t *);
int mpn_pack_detections_launch(mpn_ctx *, const float *, const float *, int, const int32_t *, const int32_t *, int, int, float *);
int mpn_select_boxes_launch(mpn_ctx *, const float *, const float *, int64_t, int, const float *, const float *, float *);
int mpn_bbox_vote_batched_launch(mpn_ctx *, const float *, const int32_t *, const int32_t *, const int32_t *, const float *, const float *, int, int,
                                 float, float, float *);
int mpn_join_rows_launch(mpn_ctx *, const __nv_bfloat16 *, const __nv_bfloat16 *, int64_t, int64_t, int64_t, int, float *);
int mpn_absmax(mpn_ctx *, const float *, int64_t, float *);
int mpn_weight_permute_half_launch(mpn_ctx *, const float *, int64_t, int, int, int, float, void *);

namespace {

struct DevBuf {           // owning device allocation
  void *p = nullptr; size_t bytes = 0;
  ~DevBuf() { if (p) cudaFree(p); }
  int ensure(mpn_ctx *ctx, size_t n) {
    if (n <= bytes) return MPN_OK;
    if (p) { cudaFree(p); p = nullptr; bytes = 0; }
    MPN_CUDA(ctx, cudaMalloc(&p, n));
    bytes = n;
    return MPN_OK;
  }
};

struct SplitBuf {         // owning hi/lo planes
  DevBuf hi, lo;
  int ensure(mpn_ctx *ctx, size_t elems) {
    MPN_TRY(hi.ensure(ctx, elems * 2 + 256));
    return lo.ensure(ctx, elems * 2 + 256);
  }
};

struct WeightDev {
  DevBuf hi, lo;          // split [Cout][K] for tensor-core convs
  DevBuf h16; float h16_scale = 0.f;   // "w16" layers (fc6 / fc7): ONE fp16 plane of w * h16_scale (a power of two)
  DevBuf f32;             // raw fp32 (Torch layout) for the direct first layer / biases
  int64_t n = 0;
};

struct LayerExec {
  mpn_layer L;
  ConvProblem prob;
  ConvPlan plan;
  bool is_direct = false;  // Cin not a multiple of 64: CUDA-core direct conv from the NCHW fp32 image
  DTensor in, out;
  // conv -> 2x2/2 max pool fusion (trunk): the conv's epilogue also writes the NEXT layer's (pool) output;
  // pool_only: the full-resolution conv output has no other reader and is not written at all.
  bool fused_pool = false, pool_only = false;
  DTensor pool_out_t;
};

int pool_out(int in, int k, int s, int p, int ceil_mode) {
  int o = ceil_mode ? (in + 2 * p - k + s - 1) / s + 1 : (in + 2 * p - k) / s + 1;
  if (ceil_mode && (o - 1) * s >= in + p) --o;
  return o;
}

}  // namespace

struct mpn_model {
  mpn_ctx *ctx = nullptr;
  mpn_model_desc d;
  std::vector<mpn_layer> trunk_layers, tower_layers;
  std::vector<mpn_tower> towers;
  std::vector<mpn_head> cls_heads;
  std::vector<std::unique_ptr<WeightDev>> weights;
  std::vector<int64_t> w_elems;
  std::vector<std::vector<float>> w_host_small;   // host copies of small arrays (first-layer filter bank / bias travel as kernel parameters)
  std::vector<int> w_prepared;     // 0 = raw only, 1 = split prepared with (Cin,kh,kw) below
  int conv_impl = 0;

  // ---- trunk state
  int tN = 0, tH = 0, tW = 0; bool trunk_valid = false;   // images, height, width the trunk is planned for
  std::vector<LayerExec> trunk_exec;
  std::map<int, DTensor> trunk_slots; std::map<int, std::unique_ptr<SplitBuf>> trunk_bufs;
  DevBuf image_dev, raw_image_dev;
  int merged_w = -1, merged_b = -1;   // weight-table entries of the concatenated head weights / biases (plan_heads)
  std::set<int> elided_slots;      // conv outputs the last trunk forward did not materialise (conv+pool fusion)
  double trunk_flops = 0, head_flops = 0;
  // max pyramids of the trunk slots that towers pool from (roi.cu): level k>=1 buffers per slot
  struct Pyramid { std::vector<std::unique_ptr<DevBuf>> lv; int nlev = 1; };   // fp32 levels 0..nlev-1
  std::map<int, Pyramid> pyramids;

  // ---- heads state
  int64_t hR = 0; bool heads_planned = false;
  struct TowerExec {
    std::unique_ptr<SplitBuf> pooled_buf; DTensor pooled; int ctot = 0;
    std::vector<LayerExec> layers; std::map<int, DTensor> slots; std::map<int, std::unique_ptr<SplitBuf>> bufs;
    int out_features = 0, col_off = 0;
    std::map<int, int> slot_fmt;           // tower slot -> 1 when it is stored as fp16 hi / lo planes (input of a "w16" Linear)
  };
  std::vector<TowerExec> tex;
  SplitBuf concat_buf; int concat_width = 0;
  std::vector<LayerExec> head_exec;     // cls heads then bbox head
  DevBuf rois_dev, boxes_dev, cls_logits, bbox_raw, scores_dev, bboxes_dev;
  DevBuf sb_dev, src_idx_dev, counts_dev, keep_idx_dev, keep_counts_dev;
  RoiJobs jobs;
  // ---- pipelined submit/wait (two slots): per-slot input staging + a private copy of the outputs, copy streams, events
  struct PipeSlot {
    DevBuf image, raw_u8, boxes, scores, bboxes, keep_idx, keep_counts;
    cudaEvent_t h2d = nullptr, compute = nullptr, done = nullptr;
    bool busy = false; int ticket = -1;
  };
  PipeSlot pipe[2];
  cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
  int next_ticket = 0;
  // ---- mpn_model_test_one: per-pass outputs, joined rows, per-class workspaces of capacity n_rows
  DevBuf to_pass_scores, to_pass_bboxes, to_new_boxes, to_scores, to_bboxes, to_sb, to_src, to_counts, to_keep, to_keep_counts, to_voted;
  // ---- detection sink (mpn_model_set_detection_sink): every detect+NMS pass also packs the image's record
  float *sink = nullptr; int64_t sink_cap = 0, sink_n = 0; int sink_top_k = 100;
  ~mpn_model() {
    for (auto &q : pipe) { if (q.h2d) cudaEventDestroy(q.h2d); if (q.compute) cudaEventDestroy(q.compute); if (q.done) cudaEventDestroy(q.done); }
    if (s_h2d) cudaStreamDestroy(s_h2d);
    if (s_d2h) cudaStreamDestroy(s_d2h);
  }
};

namespace {

int upload_weight_raw(mpn_model *m, int idx, const float *host, int64_t n) {
  WeightDev &w = *m->weights[idx];
  w.n = n;
  MPN_TRY(w.f32.ensure(m->ctx, sizeof(float) * (size_t)std::max<int64_t>(n, 1)));
  MPN_CUDA(m->ctx, cudaMemcpyAsync(w.f32.p, host, sizeof(float) * (size_t)n, cudaMemcpyHostToDevice, m->ctx->stream));
  return MPN_OK;
}

// Torch [Cout][Cin][kh][kw] -> split [Cout][kh][kw][Cin]; raw fp32 copy is then released.
int prepare_conv_weight(mpn_model *m, int idx, int Cout, int Cin, int kh, int kw) {
  mpn_ctx *ctx = m->ctx;
  MPN_CHECK_ARG(ctx, idx >= 0 && idx < (int)m->weights.size(), "layer weight index out of range");
  WeightDev &w = *m->weights[idx];
  MPN_CHECK_ARG(ctx, w.n == (int64_t)Cout * Cin * kh * kw, "weight element count does not match layer geometry");
  if (m->w_prepared[idx] == 1) return MPN_OK;
  MPN_CHECK_ARG(ctx, m->w_prepared[idx] == 0, "weight already prepared as an fp16 plane");
  const size_t elems = (size_t)w.n;
  MPN_TRY(w.hi.ensure(ctx, elems * 2 + 256));
  MPN_TRY(w.lo.ensure(ctx, elems * 2 + 256));
  MPN_TRY(mpn_weight_permute_split_launch(ctx, (const float *)w.f32.p, Cout, Cin, kh, kw, (__nv_bfloat16 *)w.hi.p,
                                          (__nv_bfloat16 *)w.lo.p));
  m->w_prepared[idx] = 1;
  // the fp32 staging copy is no longer needed (cudaFree synchronises with the split kernel)
  cudaFree(w.f32.p); w.f32.p = nullptr; w.f32.bytes = 0;
  return MPN_OK;
}

// Torch [Cout][Cin][kh][kw] -> ONE fp16 plane [Cout][kh][kw][Cin] of w * 2^e, 2^e chosen so that max|w| * 2^e lies in
// [8192, 16384) (fp16 overflows at 65504; weights 2^-27 below the largest one fall into fp16's subnormals, where they
// contribute nothing measurable); raw fp32 copy is then released.
int prepare_conv_weight_w16(mpn_model *m, int idx, int Cout, int Cin, int kh, int kw) {
  mpn_ctx *ctx = m->ctx;
  MPN_CHECK_ARG(ctx, idx >= 0 && idx < (int)m->weights.size(), "layer weight index out of range");
  WeightDev &w = *m->weights[idx];
  MPN_CHECK_ARG(ctx, w.n == (int64_t)Cout * Cin * kh * kw, "weight element count does not match layer geometry");
  if (m->w_prepared[idx] == 2) return MPN_OK;
  MPN_CHECK_ARG(ctx, m->w_prepared[idx] == 0, "weight already prepared in the split-bf16 layout");
  float amax = 0.f;
  MPN_TRY(mpn_absmax(ctx, (const float *)w.f32.p, w.n, &amax));
  MPN_CHECK_ARG(ctx, std::isfinite(amax), "weight holds a non-finite value");
  int e = 0;
  if (amax > 0.f) { (void)std::frexp(amax, &e); e = 14 - e; }          // amax = f * 2^e0, f in [0.5, 1) -> amax * 2^(14 - e0) in [8192, 16384)
  e = std::max(-60, std::min(60, e));
  w.h16_scale = std::ldexp(1.0f, e);
  MPN_TRY(w.h16.ensure(ctx, (size_t)w.n * 2 + 256));
  MPN_TRY(mpn_weight_permute_half_launch(ctx, (const float *)w.f32.p, Cout, Cin, kh, kw, w.h16_scale, w.h16.p));
  m->w_prepared[idx] = 2;
  cudaFree(w.f32.p); w.f32.p = nullptr; w.f32.bytes = 0;
  return MPN_OK;
}

DTensor make_split_view(SplitBuf &b, int64_t N, int64_t H, int64_t W, int64_t C) {
  DTensor t; t.hi = (__nv_bfloat16 *)b.hi.p; t.lo = (__nv_bfloat16 *)b.lo.p; t.N = N; t.H = H; t.W = W; t.C = C; t.ld = C;
  return t;
}

// Build the executable form of one CONV layer (weights prepared, problem + plan filled).
// flat_from: if the layer consumes a FLATTENed (h,w,c) tensor, its Linear weight [Cout][c*h*w]
// in (c,h,w) order is re-laid as a (kh=h,kw=w,Cin=c) conv weight => (h,w,c) K order.
int build_conv(mpn_model *m, LayerExec &e, const DTensor &in, DTensor out, int fh, int fw, int fc, bool per_roi = false) {
  mpn_ctx *ctx = m->ctx;
  const mpn_layer &L = e.L;
  e.in = in; e.out = out;
  ConvProblem &p = e.prob;
  p = ConvProblem();
  p.x = in; p.Cout = L.cout; p.kh = L.kh; p.kw = L.kw; p.stride = L.stride; p.pad = L.pad; p.relu = L.relu;
  p.y = out; p.y_f32_ld = out.ld;
  p.m_invariant = per_roi ? 1 : 0;
  MPN_CHECK_ARG(ctx, L.weight >= 0 && L.weight < (int)m->weights.size(), "conv layer without weight");
  // the big per-ROI Linears (fc6 / fc7) take the "w16" numerics — weight = one scaled fp16 plane, activation = fp16 hi / lo
  // planes, two tensor-core products per MAC instead of three — exactly when plan_heads gave their input fp16 planes
  const bool w16 = (in.fmt == 1);
  MPN_CHECK_ARG(ctx, !w16 || (per_roi && L.kh == 1 && L.kw == 1 && L.stride == 1 && L.pad == 0 && in.H == 1 && in.W == 1),
                "fp16 activation planes reached a layer that is not a per-ROI Linear");
  WeightDev &w = *m->weights[L.weight];
  if (w16) {
    MPN_TRY(prepare_conv_weight_w16(m, L.weight, L.cout, fc > 0 ? fc : L.cin, fc > 0 ? fh : L.kh, fc > 0 ? fw : L.kw));
    p.w16 = w.h16.p; p.w16_inv_scale = 1.0f / w.h16_scale;
  } else {
    if (fc > 0) { MPN_TRY(prepare_conv_weight(m, L.weight, L.cout, fc, fh, fw)); }
    else { MPN_TRY(prepare_conv_weight(m, L.weight, L.cout, L.cin, L.kh, L.kw)); }
    p.w_hi = (const __nv_bfloat16 *)w.hi.p; p.w_lo = (const __nv_bfloat16 *)w.lo.p;
  }
  if (L.bias >= 0) {
    MPN_CHECK_ARG(ctx, L.bias < (int)m->weights.size() && m->weights[L.bias]->n == L.cout, "bias size mismatch");
    p.bias = (const float *)m->weights[L.bias]->f32.p;
  }
  MPN_TRY(conv_tc_plan(ctx, p, e.plan));
  return MPN_OK;
}

int run_conv(mpn_model *m, LayerExec &e) {
  if (m->conv_impl == 1) return conv_ref_launch(m->ctx, e.prob);
  return conv_tc_launch(m->ctx, e.prob, e.plan);
}

// ------------------------------------------------------------------ trunk planning
int plan_trunk(mpn_model *m, int N, int H, int W) {
  mpn_ctx *ctx = m->ctx;
  m->trunk_exec.clear(); m->trunk_slots.clear();
  m->trunk_flops = 0;
  DTensor img; img.N = N; img.H = H; img.W = W; img.C = 3; img.ld = 3;   // slot 0: NCHW fp32 image (special)
  m->trunk_slots[0] = img;
  for (const mpn_layer &L : m->trunk_layers) {
    MPN_CHECK_ARG(ctx, m->trunk_slots.count(L.in_slot), "trunk layer reads an undefined slot");
    const DTensor in = m->trunk_slots[L.in_slot];
    LayerExec e; e.L = L;
    DTensor out; out.N = in.N;
    if (L.kind == MPN_LAYER_CONV) {
      MPN_CHECK_ARG(ctx, L.cin == in.C, "trunk conv cin does not match its input");
      out.H = (in.H + 2 * L.pad - L.kh) / L.stride + 1; out.W = (in.W + 2 * L.pad - L.kw) / L.stride + 1; out.C = L.cout;
    } else if (L.kind == MPN_LAYER_MAXPOOL) {
      out.H = pool_out((int)in.H, L.kh, L.stride, L.pad, L.ceil_mode);
      out.W = pool_out((int)in.W, L.kw, L.stride, L.pad, L.ceil_mode); out.C = in.C;
    } else {
      return mpn_fail(ctx, MPN_ERR_ARG, "unsupported trunk layer kind");
    }
    MPN_CHECK_ARG(ctx, out.H > 0 && out.W > 0, "trunk layer output is empty");
    MPN_CHECK_ARG(ctx, L.out_slot > 0, "trunk layers may not write slot 0");
    auto &buf = m->trunk_bufs[L.out_slot];
    if (!buf) buf.reset(new SplitBuf());
    MPN_TRY(buf->ensure(ctx, (size_t)(out.N * out.H * out.W * out.C)));
    out = make_split_view(*buf, out.N, out.H, out.W, out.C);
    if (L.kind == MPN_LAYER_CONV) {
      if (L.in_slot == 0) {
        e.is_direct = true; e.in = in; e.out = out;
        MPN_CHECK_ARG(ctx, L.weight >= 0 && m->weights[L.weight]->n == (int64_t)L.cout * L.cin * L.kh * L.kw,
                      "first-layer weight size mismatch");
      } else {
        DTensor o2 = out;
        MPN_TRY(build_conv(m, e, in, o2, 0, 0, 0));
        if (L.residual_slot >= 0) {
          MPN_CHECK_ARG(ctx, m->trunk_slots.count(L.residual_slot), "residual slot undefined");
          e.prob.res = m->trunk_slots[L.residual_slot];
        }
      }
      m->trunk_flops += 2.0 * L.cin * L.cout * L.kh * L.kw * (double)out.H * out.W * out.N;
    } else {
      e.in = in; e.out = out;
    }
    m->trunk_slots[L.out_slot] = out;
    m->trunk_exec.push_back(e);
  }
  // conv(3x3 tcgen05 kernel) immediately followed by a 2x2/2 pad-0 max pool of its output: fuse the pool into the epilogue
  {
    const char *envf = getenv("MPN_TC_FUSE_POOL");
    const bool allow = !(envf && envf[0] == '0');
    for (size_t i = 0; allow && i + 1 < m->trunk_exec.size(); ++i) {
      LayerExec &c = m->trunk_exec[i]; const LayerExec &q = m->trunk_exec[i + 1];
      if (c.L.kind != MPN_LAYER_CONV || c.is_direct || q.L.kind != MPN_LAYER_MAXPOOL) continue;
      if (q.L.in_slot != c.L.out_slot || q.L.kh != 2 || q.L.kw != 2 || q.L.stride != 2 || q.L.pad != 0) continue;
      if (c.plan.mode != 1 || c.plan.splitk != 1 || c.L.residual_slot >= 0 || (c.L.cout % 8) != 0) continue;
      if (q.out.H != (c.out.H + 1) / 2 || q.out.W != (c.out.W + 1) / 2) continue;      // floor-mode pools with odd sizes stay separate
      bool other_reader = false;
      for (size_t j = 0; j < m->trunk_exec.size(); ++j) {
        if (j == i + 1) continue;
        const mpn_layer &L2 = m->trunk_exec[j].L;
        if (j > i && (L2.in_slot == c.L.out_slot || L2.residual_slot == c.L.out_slot)) other_reader = true;
      }
      for (const mpn_tower &T : m->towers)
        for (int l = 0; l < T.n_levels; ++l) if (T.level_slot[l] == c.L.out_slot) other_reader = true;
      c.fused_pool = true; c.pool_only = !other_reader; c.pool_out_t = q.out;
    }
  }
  // max pyramids for every slot a tower pools from: levels with 2^k <= min(H, W), at most ROI_MAX_LEVELS-1 extra copies
  for (const mpn_tower &T : m->towers)
    for (int l = 0; l < T.n_levels; ++l) {
      const int slot = T.level_slot[l];
      MPN_CHECK_ARG(ctx, m->trunk_slots.count(slot) && slot > 0, "tower level reads an undefined trunk slot");
      const DTensor &f = m->trunk_slots[slot];
      mpn_model::Pyramid &P = m->pyramids[slot];
      // a level with block 2^k is only ever used for a bin window whose smaller side is >= 2^k cells; a bin of this tower
      // spans at most ceil(region_scale * map_side / pooled_side) + 1 cells of the (clipped) region, so higher levels are dead
      const double rs = T.region == 0 ? 1.0 : (T.region == 1 ? 1.5 : (T.region == 2 ? 2.0 : 4.0));
      const long long max_bin = std::min<long long>(std::min(f.H, f.W),
          (long long)std::ceil(rs * (double)std::max(f.H, f.W) / (double)std::min(T.pooled_h, T.pooled_w)) + 2);
      int nlev = 1;
      while (nlev < ROI_MAX_LEVELS && (1ll << nlev) <= max_bin) ++nlev;
      nlev = std::max(nlev, P.nlev);                                   // several towers may share the slot: keep the deepest
      P.nlev = nlev;
      P.lv.resize(nlev);
      for (int k = 0; k < nlev; ++k) {
        if (!P.lv[k]) P.lv[k].reset(new DevBuf());
        MPN_TRY(P.lv[k]->ensure(ctx, sizeof(float) * (size_t)(f.N * f.H * f.W * f.C) + 256));
      }
    }
  m->tN = N; m->tH = H; m->tW = W; m->trunk_valid = false; m->heads_planned = false;
  return MPN_OK;
}

int run_trunk(mpn_model *m, const float *image_dev) {
  mpn_ctx *ctx = m->ctx;
  m->elided_slots.clear();
  for (size_t li = 0; li < m->trunk_exec.size(); ++li) {
    LayerExec &e = m->trunk_exec[li];
    const mpn_layer &L = e.L;
    if (e.fused_pool && m->conv_impl == 0) {
      ConvProblem pf = e.prob;
      pf.pool = e.pool_out_t; pf.pool_only = e.pool_only ? 1 : 0;
      MPN_TRY(conv_tc_launch(ctx, pf, e.plan));
      if (e.pool_only) m->elided_slots.insert(L.out_slot);
      ++li;                                  // the pool layer's output is already written
      continue;
    }
    if (L.kind == MPN_LAYER_CONV) {
      if (e.is_direct) {
        const float *bias = L.bias >= 0 ? (const float *)m->weights[L.bias]->f32.p : nullptr;
        MPN_TRY(conv_direct_nchw_launch(ctx, image_dev, m->tN, L.cin, (int)e.in.H, (int)e.in.W,
                                        (const float *)m->weights[L.weight]->f32.p, bias, L.cout, L.kh, L.kw, L.stride,
                                        L.pad, L.relu, e.out,
                                        m->w_host_small[L.weight].empty() ? nullptr : m->w_host_small[L.weight].data(),
                                        (L.bias >= 0 && !m->w_host_small[L.bias].empty()) ? m->w_host_small[L.bias].data() : nullptr));
      } else {
        MPN_TRY(run_conv(m, e));
      }
    } else {
      MPN_TRY(mpn_maxpool_launch(ctx, e.in, L.kh, L.stride, L.pad, e.out));
    }
  }
  for (auto &kv : m->pyramids) {
    const DTensor &f = m->trunk_slots[kv.first];
    float *lv[ROI_MAX_LEVELS] = {nullptr};
    for (int k = 0; k < kv.second.nlev; ++k) lv[k] = (float *)kv.second.lv[k]->p;
    int too_big = 0;       // small maps (conv5): every level in one launch
    MPN_TRY(mpn_maxpyr_all_launch(ctx, f.hi, f.lo, (int)f.N, (int)f.H, (int)f.W, (int)f.C, f.ld, kv.second.nlev, lv, &too_big));
    if (!too_big) continue;
    MPN_TRY(mpn_pyr_level0_launch(ctx, f.hi, f.lo, (int)f.N, (int)f.H, (int)f.W, (int)f.C, f.ld, lv[0]));
    for (int k = 1; k < kv.second.nlev; ++k)
      MPN_TRY(mpn_maxpyr_launch(ctx, lv[k - 1], (int)f.N, (int)f.H, (int)f.W, (int)f.C, 1 << (k - 1), lv[k]));
  }
  m->trunk_valid = true;
  return MPN_OK;
}

// ------------------------------------------------------------------ heads planning
int plan_heads(mpn_model *m, int64_t R) {
  mpn_ctx *ctx = m->ctx;
  const int C = m->d.num_classes;
  m->head_flops = 0;
  m->tex.clear(); m->tex.resize(m->towers.size());
  m->jobs.n = 0;
  // concat width = sum of tower output features
  int width = 0;
  std::vector<int> feat(m->towers.size(), 0);
  for (size_t t = 0; t < m->towers.size(); ++t) {
    const mpn_tower &T = m->towers[t];
    // find the producing layer of out_slot to learn its feature count
    int f = -1;
    for (int i = 0; i < T.n_layers; ++i) {
      const mpn_layer &L = m->tower_layers[T.first_layer + i];
      if (L.out_slot == T.out_slot) f = (L.kind == MPN_LAYER_CONV) ? L.cout : -2;
    }
    MPN_CHECK_ARG(ctx, f != -1, "tower out_slot is never written");
    feat[t] = f;   // -2: resolved below (avgpool/flatten output)
  }
  // first pass to resolve shapes and features
  for (size_t t = 0; t < m->towers.size(); ++t) {
    const mpn_tower &T = m->towers[t];
    mpn_model::TowerExec &X = m->tex[t];
    X.ctot = 0;
    for (int l = 0; l < T.n_levels; ++l) {
      MPN_CHECK_ARG(ctx, m->trunk_slots.count(T.level_slot[l]) && T.level_slot[l] > 0, "tower level reads an undefined trunk slot");
      X.ctot += (int)m->trunk_slots[T.level_slot[l]].C;
    }
    X.pooled_buf.reset(new SplitBuf());
    MPN_TRY(X.pooled_buf->ensure(ctx, (size_t)R * T.pooled_h * T.pooled_w * X.ctot));
    X.pooled = make_split_view(*X.pooled_buf, R, T.pooled_h, T.pooled_w, X.ctot);
    // ROI jobs
    int ch_off = 0;
    for (int l = 0; l < T.n_levels; ++l) {
      MPN_CHECK_ARG(ctx, m->jobs.n < MAX_ROI_JOBS, "too many (tower, level) ROI jobs");
      const DTensor &f = m->trunk_slots[T.level_slot[l]];
      RoiJob &j = m->jobs.j[m->jobs.n++];
      j.H = (int)f.H; j.W = (int)f.W; j.C = (int)f.C; j.nimg = (int)f.N; j.scale = T.level_scale[l];
      MPN_TRY(mpn_ovf_flag(ctx, &j.flag));
      j.region = T.region; j.out_hi = X.pooled.hi; j.out_lo = X.pooled.lo; j.out_ld = X.ctot; j.out_ch_off = ch_off;
      j.normalize = T.normalize; j.out_fmt = 0; j.ovf = nullptr; j.tower = (int)t;
      const mpn_model::Pyramid &P = m->pyramids[T.level_slot[l]];
      j.nlev = P.nlev;
      for (int k = 0; k < ROI_MAX_LEVELS; ++k) j.lv[k] = (const float *)P.lv[std::min(k, P.nlev - 1)]->p;
      ch_off += (int)f.C;
    }
    // shape walk
    std::map<int, DTensor> shp; shp[0] = X.pooled;
    for (int i = 0; i < T.n_layers; ++i) {
      const mpn_layer &L = m->tower_layers[T.first_layer + i];
      MPN_CHECK_ARG(ctx, shp.count(L.in_slot), "tower layer reads an undefined slot");
      const DTensor in = shp[L.in_slot]; DTensor out; out.N = R;
      if (L.kind == MPN_LAYER_CONV) {
        MPN_CHECK_ARG(ctx, L.cin == in.C, "tower conv cin does not match its input");
        out.H = (in.H + 2 * L.pad - L.kh) / L.stride + 1; out.W = (in.W + 2 * L.pad - L.kw) / L.stride + 1; out.C = L.cout;
      } else if (L.kind == MPN_LAYER_FLATTEN) { out.H = 1; out.W = 1; out.C = in.H * in.W * in.C; }
      else if (L.kind == MPN_LAYER_AVGPOOL) { out.H = 1; out.W = 1; out.C = in.C; }
      else if (L.kind == MPN_LAYER_MAXPOOL) {
        out.H = pool_out((int)in.H, L.kh, L.stride, L.pad, L.ceil_mode); out.W = pool_out((int)in.W, L.kw, L.stride, L.pad, L.ceil_mode);
        out.C = in.C;
      } else return mpn_fail(ctx, MPN_ERR_ARG, "unsupported tower layer kind");
      shp[L.out_slot] = out;
    }
    // ---- plane formats of the tower's slots: the input of a "w16" Linear (fc6 / fc7: K >= 2048, >= 1024 outputs,
    // profiles/r01i_split_emulation.md) is stored as fp16 hi / lo planes by whoever produces it (the ROI kernel for slot 0,
    // the previous layer's epilogue otherwise); every reader of such a slot must be a w16 Linear (or the FLATTEN in front
    // of one), else the slot stays bf16. mpn_ctx_set_option("fc_w16", 0) / MPN_FC_W16=0 switches the scheme off.
    {
      // Default (option / environment unset): ON for single-tower graphs (Fast R-CNN: cfg 2 measures 4-5e-4 on the scores, the
      // figure the CPU emulation predicted), OFF for multi-tower graphs — the first B200 run of cfg 3 with w16 in all five
      // towers measured 2.3e-3: the class Linear reads a 4 x 4096 concat of w16 outputs and its logits are large enough that
      // the weight plane's 2^-12 becomes a visible softmax error (tests/test_model_gpu.py::test_multipathnet_full_size_cfg3).
      static const int w16_env = [] { const char *e = getenv("MPN_FC_W16"); return !e ? -1 : (e[0] == '0' ? 0 : 1); }();
      const int w16_on = ctx->opt_fc_w16 >= 0 ? ctx->opt_fc_w16 : (w16_env >= 0 ? w16_env : (m->towers.size() == 1 ? 1 : 0));
      std::map<int, int> &fmt = X.slot_fmt;
      fmt.clear();
      auto wants = [&](const mpn_layer &L) {
        if (!w16_on || L.kind != MPN_LAYER_CONV || L.residual_slot >= 0) return false;
        const DTensor &in = shp[L.in_slot];
        if (L.weight >= 0 && L.weight < (int)m->w_prepared.size() && m->w_prepared[L.weight] == 2) return true;   // the fp16 plane is what there is
        return L.kh == 1 && L.kw == 1 && L.stride == 1 && L.pad == 0 && in.H == 1 && in.W == 1 && in.C >= 2048 && L.cout >= 1024 &&
               L.weight >= 0 && L.weight < (int)m->w_prepared.size() && m->w_prepared[L.weight] != 1;
      };
      for (int i = 0; i < T.n_layers; ++i) { const mpn_layer &L = m->tower_layers[T.first_layer + i]; if (wants(L)) fmt[L.in_slot] = 1; }
      for (int pass = 0; pass < 4; ++pass) {
        for (int i = T.n_layers - 1; i >= 0; --i) {                 // a FLATTEN's output aliases its input
          const mpn_layer &L = m->tower_layers[T.first_layer + i];
          if (L.kind == MPN_LAYER_FLATTEN && fmt.count(L.out_slot) && fmt[L.out_slot]) fmt[L.in_slot] = 1;
        }
        for (int i = 0; i < T.n_layers; ++i) {                      // any other reader vetoes
          const mpn_layer &L = m->tower_layers[T.first_layer + i];
          auto veto = [&](int slot) {
            if (!fmt.count(slot) || !fmt[slot]) return;
            fmt[slot] = 0;
            for (int j = 0; j < T.n_layers; ++j) {                  // and so does the alias on the other side of a FLATTEN
              const mpn_layer &F = m->tower_layers[T.first_layer + j];
              if (F.kind == MPN_LAYER_FLATTEN && (F.in_slot == slot || F.out_slot == slot)) { fmt[F.in_slot] = 0; fmt[F.out_slot] = 0; }
            }
          };
          if (L.kind == MPN_LAYER_CONV) { if (!wants(L)) veto(L.in_slot); if (L.residual_slot >= 0) veto(L.residual_slot); }
          else if (L.kind == MPN_LAYER_FLATTEN) { if (fmt.count(L.in_slot) && fmt[L.in_slot] && !(fmt.count(L.out_slot) && fmt[L.out_slot])) veto(L.in_slot); }
          else veto(L.in_slot);
        }
        if (fmt.count(T.out_slot) && fmt[T.out_slot]) fmt[T.out_slot] = 0;      // the concat feeds the (three-product) heads
      }
    }
    MPN_CHECK_ARG(ctx, shp.count(T.out_slot), "tower out_slot undefined");
    const DTensor o = shp[T.out_slot];
    MPN_CHECK_ARG(ctx, o.H == 1 && o.W == 1, "tower output must be R x 1 x 1 x F");
    X.out_features = (int)o.C; X.col_off = width; width += (int)o.C;
  }
  for (int ji = 0; ji < m->jobs.n; ++ji) {                          // pooled tensors that feed a w16 Linear: fp16 planes
    RoiJob &j = m->jobs.j[ji];
    mpn_model::TowerExec &X = m->tex[j.tower];
    if (X.slot_fmt.count(0) && X.slot_fmt[0]) { j.out_fmt = 1; MPN_TRY(mpn_ovf_flag(ctx, &j.ovf)); X.pooled.fmt = 1; }
  }
  m->concat_width = width;
  MPN_CHECK_ARG(ctx, width % 8 == 0, "concat width must be a multiple of 8");
  MPN_TRY(m->concat_buf.ensure(ctx, (size_t)R * width));
  // second pass: allocate + build
  for (size_t t = 0; t < m->towers.size(); ++t) {
    const mpn_tower &T = m->towers[t];
    mpn_model::TowerExec &X = m->tex[t];
    X.slots.clear(); X.slots[0] = X.pooled; X.layers.clear();
    int flat_h = 0, flat_w = 0, flat_c = 0; int flat_slot = -1;
    for (int i = 0; i < T.n_layers; ++i) {
      const mpn_layer &L = m->tower_layers[T.first_layer + i];
      const DTensor in = X.slots[L.in_slot];
      LayerExec e; e.L = L;
      DTensor out; out.N = R;
      if (L.kind == MPN_LAYER_FLATTEN) {
        MPN_CHECK_ARG(ctx, in.ld == in.C, "flatten needs a dense input");
        out = in; out.H = 1; out.W = 1; out.C = in.H * in.W * in.C; out.ld = out.C;
        flat_h = (int)in.H; flat_w = (int)in.W; flat_c = (int)in.C; flat_slot = L.out_slot;
        X.slots[L.out_slot] = out; e.in = in; e.out = out; X.layers.push_back(e);
        continue;
      }
      if (L.kind == MPN_LAYER_CONV) {
        out.H = (in.H + 2 * L.pad - L.kh) / L.stride + 1; out.W = (in.W + 2 * L.pad - L.kw) / L.stride + 1; out.C = L.cout;
      } else if (L.kind == MPN_LAYER_AVGPOOL) { out.H = 1; out.W = 1; out.C = in.C; }
      else { out.H = pool_out((int)in.H, L.kh, L.stride, L.pad, L.ceil_mode); out.W = pool_out((int)in.W, L.kw, L.stride, L.pad, L.ceil_mode); out.C = in.C; }
      if (L.out_slot == T.out_slot) {      // write straight into this tower's column slice of the concat
        out.hi = (__nv_bfloat16 *)m->concat_buf.hi.p + X.col_off; out.lo = (__nv_bfloat16 *)m->concat_buf.lo.p + X.col_off;
        out.ld = width;
      } else {
        auto &buf = X.bufs[L.out_slot];
        if (!buf) buf.reset(new SplitBuf());
        MPN_TRY(buf->ensure(ctx, (size_t)(out.N * out.H * out.W * out.C)));
        DTensor v = make_split_view(*buf, out.N, out.H, out.W, out.C); out = v;
      }
      out.fmt = (X.slot_fmt.count(L.out_slot) && X.slot_fmt[L.out_slot]) ? 1 : 0;
      if (L.kind == MPN_LAYER_CONV) {
        const bool from_flat = (L.in_slot == flat_slot) && L.kh == 1 && L.kw == 1;
        MPN_TRY(build_conv(m, e, in, out, from_flat ? flat_h : 0, from_flat ? flat_w : 0, from_flat ? flat_c : 0, /*per_roi=*/true));
        if (L.residual_slot >= 0) {
          MPN_CHECK_ARG(ctx, X.slots.count(L.residual_slot), "tower residual slot undefined");
          e.prob.res = X.slots[L.residual_slot];
        }
        m->head_flops += 2.0 * (double)L.cin * L.cout * L.kh * L.kw * (double)out.H * out.W * (double)R;
      } else { e.in = in; e.out = out; }
      X.slots[L.out_slot] = out;
      X.layers.push_back(e);
    }
  }
  // heads: cls (K of them) then bbox, fp32 outputs
  const int K = (int)m->cls_heads.size();
  MPN_TRY(m->cls_logits.ensure(ctx, sizeof(float) * (size_t)K * R * C + 256));
  MPN_TRY(m->bbox_raw.ensure(ctx, sizeof(float) * (size_t)R * 4 * C + 256));
  MPN_TRY(m->scores_dev.ensure(ctx, sizeof(float) * (size_t)R * C + 256));
  MPN_TRY(m->bboxes_dev.ensure(ctx, sizeof(float) * (size_t)R * 4 * C + 256));
  m->head_exec.clear();
  auto add_head = [&](const mpn_head &h, float *out_ptr) -> int {
    MPN_CHECK_ARG(ctx, h.col_begin % 8 == 0 && h.col_begin + h.col_len <= width && h.col_len % 64 == 0, "head column range invalid");
    LayerExec e; mpn_layer L; memset(&L, 0, sizeof L);
    L.kind = MPN_LAYER_CONV; L.cin = h.col_len; L.cout = h.cout; L.kh = L.kw = 1; L.stride = 1; L.pad = 0; L.relu = 0;
    L.residual_slot = -1; L.weight = h.weight; L.bias = h.bias;
    e.L = L;
    DTensor in; in.hi = (__nv_bfloat16 *)m->concat_buf.hi.p + h.col_begin; in.lo = (__nv_bfloat16 *)m->concat_buf.lo.p + h.col_begin;
    in.N = R; in.H = 1; in.W = 1; in.C = h.col_len; in.ld = width;
    DTensor out; out.f32 = out_ptr; out.N = R; out.H = 1; out.W = 1; out.C = h.cout; out.ld = h.cout;
    MPN_TRY(build_conv(m, e, in, out, 0, 0, 0, /*per_roi=*/true));
    m->head_flops += 2.0 * (double)h.col_len * h.cout * (double)R;
    m->head_exec.push_back(e);
    return MPN_OK;
  };
  for (int k = 0; k < K; ++k) MPN_CHECK_ARG(ctx, m->cls_heads[k].cout == C, "cls head width must equal num_classes");
  MPN_CHECK_ARG(ctx, m->d.bbox_head.cout == 4 * C, "bbox head width must be 4*num_classes");
  // Optional (MPN_MERGE_HEADS=1; off by default: measured neutral, 687.8k vs 691.7k proposals/s on the same box): heads that
  // read the same columns and together have <= 128 outputs (Fast R-CNN: 21 + 84) run as ONE split-K GEMM whose reduce pass
  // scatters the column ranges to the dense per-head buffers: one launch pair instead of one per head.
  bool merged = false;
  {
    const mpn_head &b = m->d.bbox_head;
    int total = b.cout; bool same = K >= 1 && K < 7;
    for (int k = 0; k < K; ++k) { same = same && m->cls_heads[k].col_begin == b.col_begin && m->cls_heads[k].col_len == b.col_len; total += m->cls_heads[k].cout; }
    const char *envm = getenv("MPN_MERGE_HEADS");
    if (same && total <= 128 && envm && envm[0] == '1') {
      std::vector<const mpn_head *> hs;
      for (int k = 0; k < K; ++k) hs.push_back(&m->cls_heads[k]);
      hs.push_back(&b);
      if (m->merged_w < 0) {
        // concatenate the split weight planes [cout_k][col_len] and the biases once
        const size_t Kc = (size_t)b.col_len;
        m->weights.emplace_back(new WeightDev()); m->w_elems.push_back((int64_t)total * Kc); m->w_prepared.push_back(1); m->w_host_small.emplace_back();
        m->merged_w = (int)m->weights.size() - 1;
        m->weights.emplace_back(new WeightDev()); m->w_elems.push_back(total); m->w_prepared.push_back(0); m->w_host_small.emplace_back();
        m->merged_b = (int)m->weights.size() - 1;
        WeightDev &mw = *m->weights[m->merged_w], &mb = *m->weights[m->merged_b];
        mw.n = (int64_t)total * Kc; mb.n = total;
        MPN_TRY(mw.hi.ensure(ctx, mw.n * 2 + 256)); MPN_TRY(mw.lo.ensure(ctx, mw.n * 2 + 256));
        MPN_TRY(mb.f32.ensure(ctx, sizeof(float) * total));
        MPN_CUDA(ctx, cudaMemsetAsync(mb.f32.p, 0, sizeof(float) * total, ctx->stream));
        size_t row = 0;
        for (const mpn_head *h : hs) {
          MPN_TRY(prepare_conv_weight(m, h->weight, h->cout, h->col_len, 1, 1));
          const WeightDev &w = *m->weights[h->weight];
          MPN_CUDA(ctx, cudaMemcpyAsync((char *)mw.hi.p + row * Kc * 2, w.hi.p, (size_t)h->cout * Kc * 2, cudaMemcpyDeviceToDevice, ctx->stream));
          MPN_CUDA(ctx, cudaMemcpyAsync((char *)mw.lo.p + row * Kc * 2, w.lo.p, (size_t)h->cout * Kc * 2, cudaMemcpyDeviceToDevice, ctx->stream));
          if (h->bias >= 0)
            MPN_CUDA(ctx, cudaMemcpyAsync((float *)mb.f32.p + row, m->weights[h->bias]->f32.p, sizeof(float) * h->cout, cudaMemcpyDeviceToDevice, ctx->stream));
          row += (size_t)h->cout;
        }
      }
      mpn_head mh = b; mh.cout = total; mh.weight = m->merged_w; mh.bias = m->merged_b;
      MPN_TRY(add_head(mh, (float *)m->bbox_raw.p));            // the dense destination below replaces this pointer
      LayerExec &e = m->head_exec.back();
      if (e.plan.splitk > 1) {
        OutScatter sc; int c0 = 0;
        for (int k = 0; k < K; ++k) { sc.seg[sc.n++] = OutSeg{c0, c0 + C, (float *)m->cls_logits.p + (size_t)k * R * C, (long long)C}; c0 += C; }
        sc.seg[sc.n++] = OutSeg{c0, c0 + 4 * C, (float *)m->bbox_raw.p, (long long)4 * C};
        e.prob.scatter = sc;
        merged = true;
      } else {
        m->head_exec.pop_back();                                 // small K: no split-K plan, keep one GEMM per head
        m->head_flops -= 2.0 * (double)mh.col_len * mh.cout * (double)R;
      }
    }
  }
  if (!merged) {
    for (int k = 0; k < K; ++k) MPN_TRY(add_head(m->cls_heads[k], (float *)m->cls_logits.p + (size_t)k * R * C));
    MPN_TRY(add_head(m->d.bbox_head, (float *)m->bbox_raw.p));
  }
  // post-processing buffers
  MPN_TRY(m->sb_dev.ensure(ctx, sizeof(float) * (size_t)(C - 1) * R * 5 + 256));
  MPN_TRY(m->src_idx_dev.ensure(ctx, sizeof(int32_t) * (size_t)(C - 1) * R + 256));
  MPN_TRY(m->counts_dev.ensure(ctx, sizeof(int32_t) * (size_t)C + 256));
  MPN_TRY(m->keep_idx_dev.ensure(ctx, sizeof(int32_t) * (size_t)(C - 1) * R + 256));
  MPN_TRY(m->keep_counts_dev.ensure(ctx, sizeof(int32_t) * (size_t)C + 256));
  m->hR = R; m->heads_planned = true;
  return MPN_OK;
}

int run_heads(mpn_model *m, const float *rois_dev, int64_t R, bool apply_bbox_norm = true) {
  mpn_ctx *ctx = m->ctx;
  const mpn_tower &T0 = m->towers[0];
  MPN_TRY(mpn_roi_pool_fused_launch(ctx, m->jobs, rois_dev, R, T0.pooled_w, T0.pooled_h, m->d.roi_variant));
  for (size_t t = 0; t < m->towers.size(); ++t) {
    for (LayerExec &e : m->tex[t].layers) {
      switch (e.L.kind) {
        case MPN_LAYER_CONV: MPN_TRY(run_conv(m, e)); break;
        case MPN_LAYER_FLATTEN: break;
        case MPN_LAYER_AVGPOOL: MPN_TRY(mpn_avgpool_launch(ctx, e.in, e.out)); break;
        case MPN_LAYER_MAXPOOL: MPN_TRY(mpn_maxpool_launch(ctx, e.in, e.L.kh, e.L.stride, e.L.pad, e.out)); break;
        default: return mpn_fail(ctx, MPN_ERR_ARG, "bad tower layer");
      }
    }
  }
  for (LayerExec &e : m->head_exec) MPN_TRY(run_conv(m, e));
  if (m->d.has_bbox_norm && apply_bbox_norm)
    MPN_TRY(mpn_bbox_norm_launch(ctx, (float *)m->bbox_raw.p, R, 4 * m->d.num_classes, m->d.bbox_mean, m->d.bbox_std));
  return MPN_OK;
}

int ensure_trunk(mpn_model *m, int N, int H, int W) {
  if (m->trunk_exec.empty() || m->tN != N || m->tH != H || m->tW != W) MPN_TRY(plan_trunk(m, N, H, W));
  return MPN_OK;
}
int ensure_heads(mpn_model *m, int64_t R) {
  mpn_ctx *ctx = m->ctx;
  MPN_CHECK_ARG(ctx, !m->trunk_exec.empty(), "heads called before any trunk forward (ImageDetect.lua:95 asserts the same)");
  MPN_CHECK_ARG(ctx, R > 0 && R <= m->d.max_rois, "R out of range (0 < R <= max_rois)");
  if (!m->heads_planned || m->hR != R) MPN_TRY(plan_heads(m, R));
  return MPN_OK;
}

}  // namespace

// ================================================================== C ABI
extern "C" {

int mpn_model_create(mpn_ctx *ctx, const mpn_model_desc *desc, const float *const *weights, const int64_t *n_elem,
                     int32_t n_weights, mpn_model **out) {
  if (!ctx || !desc || !out) return MPN_ERR_ARG;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, desc->n_towers >= 1 && desc->n_trunk_layers >= 1 && desc->n_cls_heads >= 1, "empty model description");
  MPN_CHECK_ARG(ctx, desc->num_classes >= 2, "num_classes must be >= 2");
  MPN_CHECK_ARG(ctx, desc->roi_variant == 1 || desc->roi_variant == 2, "roi_variant must be 1 or 2");
  mpn_model *m = new mpn_model();
  m->ctx = ctx; m->d = *desc;
  m->trunk_layers.assign(desc->trunk_layers, desc->trunk_layers + desc->n_trunk_layers);
  m->tower_layers.assign(desc->tower_layers, desc->tower_layers + desc->n_tower_layers);
  m->towers.assign(desc->towers, desc->towers + desc->n_towers);
  m->cls_heads.assign(desc->cls_heads, desc->cls_heads + desc->n_cls_heads);
  m->d.trunk_layers = nullptr; m->d.tower_layers = nullptr; m->d.towers = nullptr; m->d.cls_heads = nullptr;
  for (size_t t = 1; t < m->towers.size(); ++t) {
    if (m->towers[t].pooled_w != m->towers[0].pooled_w || m->towers[t].pooled_h != m->towers[0].pooled_h) {
      delete m; return mpn_fail(ctx, MPN_ERR_ARG, "all towers must share the pooled size");
    }
  }
  m->weights.resize(n_weights); m->w_elems.assign(n_elem, n_elem + n_weights); m->w_prepared.assign(n_weights, 0);
  m->w_host_small.resize(n_weights);
  for (int i = 0; i < n_weights; ++i) {
    if (n_elem[i] <= 4096) m->w_host_small[i].assign(weights[i], weights[i] + n_elem[i]);
    m->weights[i].reset(new WeightDev());
    int r = upload_weight_raw(m, i, weights[i], n_elem[i]);
    if (r != MPN_OK) { delete m; return r; }
  }
  // the host arrays may be freed by the caller once we return
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) { delete m; return mpn_fail(ctx, MPN_ERR_CUDA, cudaGetErrorString(e)); }
  *out = m;
  return MPN_OK;
}

void mpn_model_destroy(mpn_model *m) {
  if (!m) return;
  cudaSetDevice(m->ctx->device);
  cudaStreamSynchronize(m->ctx->stream);
  if (m->s_d2h) cudaStreamSynchronize(m->s_d2h);
  delete m;
}

int mpn_model_set_conv_impl(mpn_model *m, int32_t impl) {
  if (!m) return MPN_ERR_ARG;
  MPN_CHECK_ARG(m->ctx, impl >= 0 && impl <= 2, "impl must be 0 (tcgen05), 1 (fp32 check kernel) or 2 (tcgen05 without conv+pool fusion)");
  m->conv_impl = impl;
  return MPN_OK;
}

int mpn_model_last_flops(const mpn_model *m, double *trunk_flops, double *head_flops) {
  if (!m) return MPN_ERR_ARG;
  if (trunk_flops) *trunk_flops = m->trunk_flops;
  if (head_flops) *head_flops = m->head_flops;
  return MPN_OK;
}

int mpn_model_trunk_batch_dev(mpn_model *m, const float *images_dev, int32_t N, int32_t H, int32_t W) {
  if (!m) return MPN_ERR_ARG;
  mpn_ctx *ctx = m->ctx;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, N >= 1 && N <= MPN_MAX_BATCH, "batch size N must be in 1..MPN_MAX_BATCH");
  MPN_CHECK_ARG(ctx, images_dev && H > 0 && W > 0 && H <= m->d.max_h && W <= m->d.max_w, "image missing or larger than max_h x max_w");
  MPN_TRY(ensure_trunk(m, N, H, W));
  return run_trunk(m, images_dev);
}

int mpn_model_trunk_dev(mpn_model *m, const float *image_dev, int32_t H, int32_t W) {
  return mpn_model_trunk_batch_dev(m, image_dev, 1, H, W);
}

int mpn_model_trunk_batch(mpn_model *m, const float *images, int32_t N, int32_t H, int32_t W) {
  if (!m) return MPN_ERR_ARG;
  mpn_ctx *ctx = m->ctx;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, images && N >= 1 && N <= MPN_MAX_BATCH && H > 0 && W > 0, "images missing or batch size outside 1..MPN_MAX_BATCH");
  const size_t bytes = sizeof(float) * 3 * (size_t)N * H * W;
  MPN_TRY(m->image_dev.ensure(ctx, bytes));
  MPN_CUDA(ctx, cudaMemcpyAsync(m->image_dev.p, images, bytes, cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(mpn_model_trunk_batch_dev(m, (const float *)m->image_dev.p, N, H, W));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MPN_OK;
}

int mpn_model_trunk(mpn_model *m, const float *image, int32_t H, int32_t W) {
  if (!m) return MPN_ERR_ARG;
  mpn_ctx *ctx = m->ctx;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, image && H > 0 && W > 0, "image missing");
  const size_t bytes = sizeof(float) * 3 * (size_t)H * W;
  MPN_TRY(m->image_dev.ensure(ctx, bytes));
  MPN_CUDA(ctx, cudaMemcpyAsync(m->image_dev.p, image, bytes, cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(mpn_model_trunk_dev(m, (const float *)m->image_dev.p, H, W));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MPN_OK;
}

int mpn_model_trunk_image(mpn_model *m, const float *im, int32_t H0, int32_t W0, const mpn_image_transform *tf,
                          double scale, double max_size, double *im_scale, int32_t *h_out, int32_t *w_out) {
  if (!m) return MPN_ERR_ARG;
  mpn_ctx *ctx = m->ctx;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, im && tf && H0 > 0 && W0 > 0, "image or transformer missing");
  int32_t h = 0, w = 0; double s = 0;
  MPN_CHECK_ARG(ctx, mpn_get_images_size_impl(H0, W0, scale, max_size, &h, &w, &s) == MPN_OK && h > 0 && w > 0, "bad scale / max_size");
  MPN_CHECK_ARG(ctx, h <= m->d.max_h && w <= m->d.max_w, "scaled image larger than max_h x max_w");
  const size_t braw = sizeof(float) * 3 * (size_t)H0 * W0, bimg = sizeof(float) * 3 * (size_t)h * w;
  MPN_TRY(m->raw_image_dev.ensure(ctx, braw));
  MPN_TRY(m->image_dev.ensure(ctx, bimg));
  MPN_CUDA(ctx, cudaMemcpyAsync(m->raw_image_dev.p, im, braw, cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(mpn_get_images_launch(ctx, (const float *)m->raw_image_dev.p, H0, W0, tf, h, w, (float *)m->image_dev.p));
  MPN_TRY(mpn_model_trunk_dev(m, (const float *)m->image_dev.p, h, w));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (im_scale) *im_scale = s;
  if (h_out) *h_out = h;
  if (w_out) *w_out = w;
  return MPN_OK;
}

int mpn_model_heads_dev(mpn_model *m, const float *rois_dev, int64_t R, float *cls_out_dev, float *bbox_out_dev) {
  if (!m) return MPN_ERR_ARG;
  mpn_ctx *ctx = m->ctx;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, m->trunk_valid, "heads called before a trunk forward");
  MPN_TRY(ensure_heads(m, R));
  MPN_TRY(run_heads(m, rois_dev, R));
  const int C = m->d.num_classes, K = (int)m->cls_heads.size();
  if (cls_out_dev) {
    if (K == 1) {   // a single head's own output: what the Linear produced (the same rule as detect: any softmax is applied there)
      MPN_CUDA(ctx, cudaMemcpyAsync(cls_out_dev, m->cls_logits.p, sizeof(float) * (size_t)R * C, cudaMemcpyDeviceToDevice, ctx->stream));
    } else {   // integral head: the model's own output is the mean of K softmaxes
      MPN_TRY(mpn_softmax_mean_launch(ctx, (const float *)m->cls_logits.p, R, C, K, 1, cls_out_dev));
    }
  }
  if (bbox_out_dev)
    MPN_CUDA(ctx, cudaMemcpyAsync(bbox_out_dev, m->bbox_raw.p, sizeof(float) * (size_t)R * 4 * C, cudaMemcpyDeviceToDevice, ctx->stream));
  return MPN_OK;
}

int mpn_model_heads(mpn_model *m, const float *rois, int64_t R, float *cls_out, float *bbox_out) {
  if (!m) return MPN_ERR_ARG;
  mpn_ctx *ctx = m->ctx;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, rois && R > 0, "rois missing");
  const int C = m->d.num_classes;
  MPN_TRY(m->rois_dev.ensure(ctx, sizeof(float) * 5 * (size_t)R));
  MPN_CUDA(ctx, cudaMemcpyAsync(m->rois_dev.p, rois, sizeof(float) * 5 * (size_t)R, cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(ensure_heads(m, R));
  MPN_TRY(mpn_model_heads_dev(m, (const float *)m->rois_dev.p, R, (float *)m->scores_dev.p, nullptr));
  if (cls_out) MPN_CUDA(ctx, cudaMemcpyAsync(cls_out, m->scores_dev.p, sizeof(float) * (size_t)R * C, cudaMemcpyDeviceToHost, ctx->stream));
  if (bbox_out) MPN_CUDA(ctx, cudaMemcpyAsync(bbox_out, m->bbox_raw.p, sizeof(float) * (size_t)R * 4 * C, cudaMemcpyDeviceToHost, ctx->stream));
  MPN_TRY(mpn_ovf_copy_async(ctx, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return mpn_ovf_test(ctx);
}

// one detect pass on the cached trunk features: project_im_rois -> heads -> scores (softmax / integral mean) | BBoxNorm +
// decode (+ clamp) into caller-chosen buffers (ImageDetect.lua:161-192 after getImages; Tester_FRCNN.lua:75-78 clamp)
static int run_detect_pass(mpn_model *m, const float *boxes_dev, int64_t R, float im_scale, int do_clamp, float W0, float H0,
                           float *scores_dst, float *bboxes_dst) {
  mpn_ctx *ctx = m->ctx;
  const int C = m->d.num_classes, K = (int)m->cls_heads.size();
  MPN_TRY(ensure_heads(m, R));
  MPN_TRY(m->rois_dev.ensure(ctx, sizeof(float) * 5 * (size_t)R));
  MPN_TRY(mpn_project_rois_launch(ctx, boxes_dev, R, im_scale, (float *)m->rois_dev.p));
  MPN_TRY(run_heads(m, (const float *)m->rois_dev.p, R, /*apply_bbox_norm=*/false));
  // class_values: softmax unless model.noSoftMax; an integral head IS its mean of softmaxes (noSoftMax=true).
  // One launch: softmax (+mean) | BBoxNorm + decode (+ clamp to the image for the NMS path, Tester_FRCNN.lua:75-78)
  const int do_softmax = (K > 1) ? 1 : (m->d.no_softmax ? 0 : 1);
  return mpn_detect_tail_launch(ctx, (const float *)m->cls_logits.p, R, C, K, do_softmax, scores_dst, (const float *)m->bbox_raw.p, boxes_dev,
                                do_clamp, W0, H0, bboxes_dst, m->d.has_bbox_norm ? 1 : 0, m->d.bbox_mean, m->d.bbox_std);
}

// shared tail: heads -> scores (softmax / integral mean) -> decode (+clamp) [-> gather -> NMS]
static int detect_tail_dev(mpn_model *m, const float *boxes_dev, int64_t R, float im_scale, int do_nms, float W0,
                           float H0, float score_thresh, float nms_thr) {
  mpn_ctx *ctx = m->ctx;
  const int C = m->d.num_classes;
  MPN_TRY(ensure_heads(m, R));
  MPN_TRY(run_detect_pass(m, boxes_dev, R, im_scale, do_nms, W0, H0, (float *)m->scores_dev.p, (float *)m->bboxes_dev.p));
  if (do_nms) {
    MPN_TRY(mpn_gather_scored_launch(ctx, (const float *)m->scores_dev.p, (const float *)m->bboxes_dev.p, (int)R, C,
                                     score_thresh, (float *)m->sb_dev.p, (int32_t *)m->src_idx_dev.p, (int32_t *)m->counts_dev.p));
    MPN_TRY(mpn_nms_launch(ctx, (const float *)m->sb_dev.p, (int)R, C - 1, (const int32_t *)m->counts_dev.p,
                           (const int32_t *)m->src_idx_dev.p, nms_thr, (int32_t *)m->keep_idx_dev.p,
                           (int32_t *)m->keep_counts_dev.p));
    if (m->sink) {     // keep_top_k + fixed-size record of this image, appended to the caller's sink (SURVEY 8e)
      MPN_CHECK_ARG(ctx, m->sink_n < m->sink_cap, "detection sink is full (mpn_model_set_detection_sink capacity)");
      MPN_TRY(mpn_pack_detections_launch(ctx, (const float *)m->scores_dev.p, (const float *)m->bboxes_dev.p, C,
                                         (const int32_t *)m->keep_idx_dev.p, (const int32_t *)m->keep_counts_dev.p, (int)R,
                                         m->sink_top_k, m->sink + (size_t)m->sink_n * MPN_REC_FLOATS));
      ++m->sink_n;
    }
  }
  return MPN_OK;
}

int mpn_model_detect(mpn_model *m, const float *image, int32_t H, int32_t W, const float *boxes, int64_t R,
                     float im_scale, int32_t recompute_features, float *scores, float *bboxes) {
  if (!m) return MPN_ERR_ARG;
  mpn_ctx *ctx = m->ctx;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, boxes && R > 0, "boxes missing");
  const int C = m->d.num_classes;
  if (recompute_features) {
    MPN_CHECK_ARG(ctx, image, "image missing");
    const size_t bytes = sizeof(float) * 3 * (size_t)H * W;
    MPN_TRY(m->image_dev.ensure(ctx, bytes));
    MPN_CUDA(ctx, cudaMemcpyAsync(m->image_dev.p, image, bytes, cudaMemcpyHostToDevice, ctx->stream));
    MPN_TRY(mpn_model_trunk_dev(m, (const float *)m->image_dev.p, H, W));
  } else {
    MPN_CHECK_ARG(ctx, m->trunk_valid, "recompute_features=false needs cached trunk features (ImageDetect.lua:109-111)");
  }
  MPN_TRY(m->boxes_dev.ensure(ctx, sizeof(float) * 4 * (size_t)R));
  MPN_CUDA(ctx, cudaMemcpyAsync(m->boxes_dev.p, boxes, sizeof(float) * 4 * (size_t)R, cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(detect_tail_dev(m, (const float *)m->boxes_dev.p, R, im_scale, 0, 0.f, 0.f, 0.f, 0.f));
  if (scores) MPN_CUDA(ctx, cudaMemcpyAsync(scores, m->scores_dev.p, sizeof(float) * (size_t)R * C, cudaMemcpyDeviceToHost, ctx->stream));
  if (bboxes) MPN_CUDA(ctx, cudaMemcpyAsync(bboxes, m->bboxes_dev.p, sizeof(float) * (size_t)R * 4 * C, cudaMemcpyDeviceToHost, ctx->stream));
  MPN_TRY(mpn_ovf_copy_async(ctx, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return mpn_ovf_test(ctx);
}

int mpn_model_detect_nms_dev(mpn_model *m, const float *image_dev, int32_t H, int32_t W, const float *boxes_dev,
                             int64_t R, float im_scale, float W0, float H0, float score_thresh, float nms_thr,
                             float *scores_dev, float *bboxes_dev, int32_t *keep_idx_dev, int32_t *keep_counts_dev) {
  if (!m) return MPN_ERR_ARG;
  mpn_ctx *ctx = m->ctx;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, image_dev && boxes_dev && R > 0, "image/boxes missing");
  const int C = m->d.num_classes;
  MPN_TRY(mpn_model_trunk_dev(m, image_dev, H, W));
  MPN_TRY(detect_tail_dev(m, boxes_dev, R, im_scale, 1, W0, H0, score_thresh, nms_thr));
  if (scores_dev) MPN_CUDA(ctx, cudaMemcpyAsync(scores_dev, m->scores_dev.p, sizeof(float) * (size_t)R * C, cudaMemcpyDeviceToDevice, ctx->stream));
  if (bboxes_dev) MPN_CUDA(ctx, cudaMemcpyAsync(bboxes_dev, m->bboxes_dev.p, sizeof(float) * (size_t)R * 4 * C, cudaMemcpyDeviceToDevice, ctx->stream));
  if (keep_idx_dev) MPN_CUDA(ctx, cudaMemcpyAsync(keep_idx_dev, m->keep_idx_dev.p, sizeof(int32_t) * (size_t)(C - 1) * R, cudaMemcpyDeviceToDevice, ctx->stream));
  if (keep_counts_dev) MPN_CUDA(ctx, cudaMemcpyAsync(keep_counts_dev, m->keep_counts_dev.p, sizeof(int32_t) * (size_t)(C - 1), cudaMemcpyDeviceToDevice, ctx->stream));
  return MPN_OK;
}

int mpn_model_detect_nms(mpn_model *m, const float *image, int32_t H, int32_t W, const float *boxes, int64_t R,
                         float im_scale, float W0, float H0, float score_thresh, float nms_thr, float *scores,
                         float *bboxes, int32_t *keep_idx, int32_t *keep_counts) {
  if (!m) return MPN_ERR_ARG;
  mpn_ctx *ctx = m->ctx;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, image && boxes && R > 0, "image/boxes missing");
  const int C = m->d.num_classes;
  const size_t bytes = sizeof(float) * 3 * (size_t)H * W;
  MPN_TRY(m->image_dev.ensure(ctx, bytes));
  MPN_TRY(m->boxes_dev.ensure(ctx, sizeof(float) * 4 * (size_t)R));
  MPN_CUDA(ctx, cudaMemcpyAsync(m->image_dev.p, image, bytes, cudaMemcpyHostToDevice, ctx->stream));
  MPN_CUDA(ctx, cudaMemcpyAsync(m->boxes_dev.p, boxes, sizeof(float) * 4 * (size_t)R, cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(mpn_model_trunk_dev(m, (const float *)m->image_dev.p, H, W));
  MPN_TRY(detect_tail_dev(m, (const float *)m->boxes_dev.p, R, im_scale, 1, W0, H0, score_thresh, nms_thr));
  if (scores) MPN_CUDA(ctx, cudaMemcpyAsync(scores, m->scores_dev.p, sizeof(float) * (size_t)R * C, cudaMemcpyDeviceToHost, ctx->stream));
  if (bboxes) MPN_CUDA(ctx, cudaMemcpyAsync(bboxes, m->bboxes_dev.p, sizeof(float) * (size_t)R * 4 * C, cudaMemcpyDeviceToHost, ctx->stream));
  if (keep_idx) MPN_CUDA(ctx, cudaMemcpyAsync(keep_idx, m->keep_idx_dev.p, sizeof(int32_t) * (size_t)(C - 1) * R, cudaMemcpyDeviceToHost, ctx->stream));
  if (keep_counts) MPN_CUDA(ctx, cudaMemcpyAsync(keep_counts, m->keep_counts_dev.p, sizeof(int32_t) * (size_t)(C - 1), cudaMemcpyDeviceToHost, ctx->stream));
  MPN_TRY(mpn_ovf_copy_async(ctx, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return mpn_ovf_test(ctx);
}

// ---- N images in one pass: host-side validation of the batch description (nothing is launched before it passes)
static int batch_desc(mpn_model *m, int32_t N, const int64_t *offs, const float *im_scale, const float *W0, const float *H0,
                      MpnBatch &b, int &cap) {
  mpn_ctx *ctx = m->ctx;
  MPN_CHECK_ARG(ctx, N >= 1 && N <= MPN_MAX_BATCH, "batch size N must be in 1..MPN_MAX_BATCH");
  MPN_CHECK_ARG(ctx, offs && im_scale && W0 && H0, "img_offsets / im_scale / W0 / H0 missing");
  MPN_CHECK_ARG(ctx, offs[0] == 0, "img_offsets[0] must be 0");
  memset(&b, 0, sizeof b);
  b.n = N; cap = 0;
  for (int i = 0; i < N; ++i) {
    MPN_CHECK_ARG(ctx, offs[i + 1] - offs[i] >= 1, "every image needs at least one proposal (img_offsets strictly increasing)");
    MPN_CHECK_ARG(ctx, offs[i + 1] <= m->d.max_rois, "R_total out of range (R_total <= max_rois)");
    b.off[i] = (int)offs[i]; b.scale[i] = im_scale[i]; b.W0[i] = W0[i]; b.H0[i] = H0[i];
    cap = std::max(cap, (int)(offs[i + 1] - offs[i]));
  }
  b.off[N] = (int)offs[N];
  return MPN_OK;
}

// trunk over the batch, heads over all R_total rows, per-image clamp, gather + NMS over N x (C-1) segments of capacity `cap`
// (segment i * (C-1) + j - 1 at sb / keep_idx_dev + seg * cap), one record per image into the sink. Results stay in the
// model's buffers.
static int detect_nms_batch_core(mpn_model *m, const float *images_dev, int32_t N, int32_t H, int32_t W, const float *boxes_dev,
                                 const MpnBatch &b, int cap, float score_thresh, float nms_thr) {
  mpn_ctx *ctx = m->ctx;
  const int C = m->d.num_classes, K = (int)m->cls_heads.size();
  const int64_t R = b.off[N];
  const int nseg = N * (C - 1);
  MPN_CHECK_ARG(ctx, !m->sink || m->sink_n + N <= m->sink_cap, "detection sink is full (mpn_model_set_detection_sink capacity)");
  MPN_TRY(mpn_model_trunk_batch_dev(m, images_dev, N, H, W));
  MPN_TRY(ensure_heads(m, R));
  MPN_TRY(m->rois_dev.ensure(ctx, sizeof(float) * 5 * (size_t)R));
  MPN_TRY(m->sb_dev.ensure(ctx, sizeof(float) * (size_t)nseg * cap * 5 + 256));
  MPN_TRY(m->src_idx_dev.ensure(ctx, sizeof(int32_t) * (size_t)nseg * cap + 256));
  MPN_TRY(m->counts_dev.ensure(ctx, sizeof(int32_t) * (size_t)nseg + 256));
  MPN_TRY(m->keep_idx_dev.ensure(ctx, sizeof(int32_t) * (size_t)nseg * cap + 256));
  MPN_TRY(m->keep_counts_dev.ensure(ctx, sizeof(int32_t) * (size_t)nseg + 256));
  MPN_TRY(mpn_project_rois_batch_launch(ctx, boxes_dev, R, b, (float *)m->rois_dev.p));
  MPN_TRY(run_heads(m, (const float *)m->rois_dev.p, R, /*apply_bbox_norm=*/false));
  const int do_softmax = (K > 1) ? 1 : (m->d.no_softmax ? 0 : 1);
  MPN_TRY(mpn_detect_tail_batch_launch(ctx, (const float *)m->cls_logits.p, R, C, K, do_softmax, (float *)m->scores_dev.p,
                                       (const float *)m->bbox_raw.p, boxes_dev, b, (float *)m->bboxes_dev.p, m->d.has_bbox_norm ? 1 : 0,
                                       m->d.bbox_mean, m->d.bbox_std));
  MPN_TRY(mpn_gather_scored_batch_launch(ctx, (const float *)m->scores_dev.p, (const float *)m->bboxes_dev.p, C, score_thresh, b, cap,
                                         (float *)m->sb_dev.p, (int32_t *)m->src_idx_dev.p, (int32_t *)m->counts_dev.p));
  MPN_TRY(mpn_nms_launch(ctx, (const float *)m->sb_dev.p, cap, nseg, (const int32_t *)m->counts_dev.p, (const int32_t *)m->src_idx_dev.p,
                         nms_thr, (int32_t *)m->keep_idx_dev.p, (int32_t *)m->keep_counts_dev.p));
  if (m->sink) {
    for (int i = 0; i < N; ++i) {
      MPN_TRY(mpn_pack_detections_launch(ctx, (const float *)m->scores_dev.p + (size_t)b.off[i] * C,
                                         (const float *)m->bboxes_dev.p + (size_t)b.off[i] * 4 * C, C,
                                         (const int32_t *)m->keep_idx_dev.p + (size_t)i * (C - 1) * cap,
                                         (const int32_t *)m->keep_counts_dev.p + (size_t)i * (C - 1), cap, m->sink_top_k,
                                         m->sink + (size_t)m->sink_n * MPN_REC_FLOATS));
      ++m->sink_n;
    }
  }
  return MPN_OK;
}

// results of detect_nms_batch_core -> the caller's buffers (device or host, by `kind`): keep lists repacked from capacity
// `cap` per segment to R_i per segment, image i's block at (C-1) * off[i]
static int detect_nms_batch_copy_out(mpn_model *m, const MpnBatch &b, int cap, cudaMemcpyKind kind, float *scores, float *bboxes,
                                     int32_t *keep_idx, int32_t *keep_counts) {
  mpn_ctx *ctx = m->ctx;
  const int C = m->d.num_classes, N = b.n;
  const int64_t R = b.off[N];
  if (scores) MPN_CUDA(ctx, cudaMemcpyAsync(scores, m->scores_dev.p, sizeof(float) * (size_t)R * C, kind, ctx->stream));
  if (bboxes) MPN_CUDA(ctx, cudaMemcpyAsync(bboxes, m->bboxes_dev.p, sizeof(float) * (size_t)R * 4 * C, kind, ctx->stream));
  if (keep_idx)
    for (int i = 0; i < N; ++i) {
      const size_t Ri = (size_t)(b.off[i + 1] - b.off[i]);
      MPN_CUDA(ctx, cudaMemcpy2DAsync(keep_idx + (size_t)(C - 1) * b.off[i], sizeof(int32_t) * Ri,
                                      (const int32_t *)m->keep_idx_dev.p + (size_t)i * (C - 1) * cap, sizeof(int32_t) * (size_t)cap,
                                      sizeof(int32_t) * Ri, (size_t)(C - 1), kind, ctx->stream));
    }
  if (keep_counts)
    MPN_CUDA(ctx, cudaMemcpyAsync(keep_counts, m->keep_counts_dev.p, sizeof(int32_t) * (size_t)N * (C - 1), kind, ctx->stream));
  return MPN_OK;
}

int mpn_model_detect_nms_batch_dev(mpn_model *m, const float *images_dev, int32_t N, int32_t H, int32_t W, const float *boxes_dev,
                                   const int64_t *img_offsets, const float *im_scale, const float *W0, const float *H0,
                                   float score_thresh, float nms_thr, float *scores_dev, float *bboxes_dev, int32_t *keep_idx_dev,
                                   int32_t *keep_counts_dev) {
  if (!m) return MPN_ERR_ARG;
  mpn_ctx *ctx = m->ctx;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, images_dev && boxes_dev, "images/boxes missing");
  MpnBatch b; int cap = 0;
  MPN_TRY(batch_desc(m, N, img_offsets, im_scale, W0, H0, b, cap));
  if (N == 1)        // one image: the single-image path, byte for byte
    return mpn_model_detect_nms_dev(m, images_dev, H, W, boxes_dev, img_offsets[1], im_scale[0], W0[0], H0[0], score_thresh, nms_thr,
                                    scores_dev, bboxes_dev, keep_idx_dev, keep_counts_dev);
  MPN_TRY(detect_nms_batch_core(m, images_dev, N, H, W, boxes_dev, b, cap, score_thresh, nms_thr));
  return detect_nms_batch_copy_out(m, b, cap, cudaMemcpyDeviceToDevice, scores_dev, bboxes_dev, keep_idx_dev, keep_counts_dev);
}

int mpn_model_detect_nms_batch(mpn_model *m, const float *images, int32_t N, int32_t H, int32_t W, const float *boxes,
                               const int64_t *img_offsets, const float *im_scale, const float *W0, const float *H0, float score_thresh,
                               float nms_thr, float *scores, float *bboxes, int32_t *keep_idx, int32_t *keep_counts) {
  if (!m) return MPN_ERR_ARG;
  mpn_ctx *ctx = m->ctx;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, images && boxes && H > 0 && W > 0, "images/boxes missing");
  MpnBatch b; int cap = 0;
  MPN_TRY(batch_desc(m, N, img_offsets, im_scale, W0, H0, b, cap));
  if (N == 1)
    return mpn_model_detect_nms(m, images, H, W, boxes, img_offsets[1], im_scale[0], W0[0], H0[0], score_thresh, nms_thr, scores, bboxes,
                                keep_idx, keep_counts);
  const int64_t R = b.off[N];
  const size_t bytes = sizeof(float) * 3 * (size_t)N * H * W;
  MPN_TRY(m->image_dev.ensure(ctx, bytes));
  MPN_TRY(m->boxes_dev.ensure(ctx, sizeof(float) * 4 * (size_t)R));
  MPN_CUDA(ctx, cudaMemcpyAsync(m->image_dev.p, images, bytes, cudaMemcpyHostToDevice, ctx->stream));
  MPN_CUDA(ctx, cudaMemcpyAsync(m->boxes_dev.p, boxes, sizeof(float) * 4 * (size_t)R, cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(detect_nms_batch_core(m, (const float *)m->image_dev.p, N, H, W, (const float *)m->boxes_dev.p, b, cap, score_thresh, nms_thr));
  MPN_TRY(detect_nms_batch_copy_out(m, b, cap, cudaMemcpyDeviceToHost, scores, bboxes, keep_idx, keep_counts));
  MPN_TRY(mpn_ovf_copy_async(ctx, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return mpn_ovf_test(ctx);
}

// the pipeline slot the next ticket uses (its copy streams and events created on first use); fails while it is in flight
static int pipe_slot(mpn_model *m, mpn_model::PipeSlot *&slot) {
  mpn_ctx *ctx = m->ctx;
  mpn_model::PipeSlot &q = m->pipe[m->next_ticket & 1];
  if (q.busy) return mpn_fail(ctx, MPN_ERR_STATE, "two submissions are already in flight: call mpn_model_detect_nms_wait first");
  if (!m->s_h2d) {
    MPN_CUDA(ctx, cudaStreamCreateWithFlags(&m->s_h2d, cudaStreamNonBlocking));
    MPN_CUDA(ctx, cudaStreamCreateWithFlags(&m->s_d2h, cudaStreamNonBlocking));
  }
  if (!q.h2d) {
    MPN_CUDA(ctx, cudaEventCreateWithFlags(&q.h2d, cudaEventDisableTiming));
    MPN_CUDA(ctx, cudaEventCreateWithFlags(&q.compute, cudaEventDisableTiming));
    MPN_CUDA(ctx, cudaEventCreateWithFlags(&q.done, cudaEventDisableTiming));
  }
  slot = &q;
  return MPN_OK;
}

// after the slot's kernels: its private outputs (R rows, n_img x (C-1) keep counts) -> the caller's host buffers on the
// device->host stream; the slot is in flight until mpn_model_detect_nms_wait(*ticket)
static int pipe_finish(mpn_model *m, mpn_model::PipeSlot &q, int64_t R, int n_img, float *scores, float *bboxes, int32_t *keep_idx,
                       int32_t *keep_counts, int32_t *ticket) {
  mpn_ctx *ctx = m->ctx;
  const int C = m->d.num_classes;
  MPN_CUDA(ctx, cudaEventRecord(q.compute, ctx->stream));
  MPN_CUDA(ctx, cudaStreamWaitEvent(m->s_d2h, q.compute, 0));
  if (scores) MPN_CUDA(ctx, cudaMemcpyAsync(scores, q.scores.p, sizeof(float) * (size_t)R * C, cudaMemcpyDeviceToHost, m->s_d2h));
  if (bboxes) MPN_CUDA(ctx, cudaMemcpyAsync(bboxes, q.bboxes.p, sizeof(float) * (size_t)R * 4 * C, cudaMemcpyDeviceToHost, m->s_d2h));
  if (keep_idx) MPN_CUDA(ctx, cudaMemcpyAsync(keep_idx, q.keep_idx.p, sizeof(int32_t) * (size_t)(C - 1) * R, cudaMemcpyDeviceToHost, m->s_d2h));
  if (keep_counts)
    MPN_CUDA(ctx, cudaMemcpyAsync(keep_counts, q.keep_counts.p, sizeof(int32_t) * (size_t)n_img * (C - 1), cudaMemcpyDeviceToHost, m->s_d2h));
  MPN_TRY(mpn_ovf_copy_async(ctx, m->s_d2h));
  MPN_CUDA(ctx, cudaEventRecord(q.done, m->s_d2h));
  q.busy = true; q.ticket = m->next_ticket;
  *ticket = m->next_ticket++;
  return MPN_OK;
}

// image != null: the transformed + scaled fp32 image (H x W); else raw_u8: the RAW H0 x W0 x 3 byte image, transformed and
// scaled on the device (get_images_kernel) to the size getImages prescribes
static int submit_common(mpn_model *m, const float *image, int32_t H, int32_t W, const uint8_t *raw_u8, int32_t H0r, int32_t W0r,
                         const mpn_image_transform *tf, double scale, double max_size, const float *boxes, int64_t R, float im_scale,
                         float W0, float H0, float score_thresh, float nms_thr, float *scores, float *bboxes, int32_t *keep_idx,
                         int32_t *keep_counts, int32_t *ticket) {
  mpn_ctx *ctx = m->ctx;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, (image || raw_u8) && boxes && R > 0 && ticket, "image/boxes/ticket missing");
  const int C = m->d.num_classes;
  mpn_model::PipeSlot *qp = nullptr;
  MPN_TRY(pipe_slot(m, qp));
  mpn_model::PipeSlot &q = *qp;
  if (raw_u8) {
    MPN_CHECK_ARG(ctx, tf && H0r > 0 && W0r > 0, "raw image: transformer / size missing");
    double s = 0;
    MPN_CHECK_ARG(ctx, mpn_get_images_size_impl(H0r, W0r, scale, max_size, &H, &W, &s) == MPN_OK && H > 0 && W > 0, "bad scale / max_size");
    MPN_CHECK_ARG(ctx, H <= m->d.max_h && W <= m->d.max_w, "scaled image larger than max_h x max_w");
    im_scale = (float)s; W0 = (float)W0r; H0 = (float)H0r;          // clamp to the ORIGINAL image (Tester_FRCNN.lua:75-78)
  }
  const size_t img_bytes = sizeof(float) * 3 * (size_t)H * W;
  MPN_TRY(q.image.ensure(ctx, img_bytes));
  MPN_TRY(q.boxes.ensure(ctx, sizeof(float) * 4 * (size_t)R));
  MPN_TRY(q.scores.ensure(ctx, sizeof(float) * (size_t)R * C));
  MPN_TRY(q.bboxes.ensure(ctx, sizeof(float) * (size_t)R * 4 * C));
  MPN_TRY(q.keep_idx.ensure(ctx, sizeof(int32_t) * (size_t)(C - 1) * R));
  MPN_TRY(q.keep_counts.ensure(ctx, sizeof(int32_t) * (size_t)(C - 1)));
  // inputs: the slot's previous occupant was waited for (busy == false), so its staging buffers are free
  if (raw_u8) {
    MPN_TRY(q.raw_u8.ensure(ctx, (size_t)H0r * W0r * 3));
    MPN_CUDA(ctx, cudaMemcpyAsync(q.raw_u8.p, raw_u8, (size_t)H0r * W0r * 3, cudaMemcpyHostToDevice, m->s_h2d));
  } else {
    MPN_CUDA(ctx, cudaMemcpyAsync(q.image.p, image, img_bytes, cudaMemcpyHostToDevice, m->s_h2d));
  }
  MPN_CUDA(ctx, cudaMemcpyAsync(q.boxes.p, boxes, sizeof(float) * 4 * (size_t)R, cudaMemcpyHostToDevice, m->s_h2d));
  MPN_CUDA(ctx, cudaEventRecord(q.h2d, m->s_h2d));
  MPN_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, q.h2d, 0));
  if (raw_u8) MPN_TRY(mpn_get_images_u8_launch(ctx, (const uint8_t *)q.raw_u8.p, H0r, W0r, tf, H, W, (float *)q.image.p));
  MPN_TRY(mpn_model_detect_nms_dev(m, (const float *)q.image.p, H, W, (const float *)q.boxes.p, R, im_scale, W0, H0, score_thresh,
                                   nms_thr, scores ? (float *)q.scores.p : nullptr, bboxes ? (float *)q.bboxes.p : nullptr,
                                   keep_idx ? (int32_t *)q.keep_idx.p : nullptr, keep_counts ? (int32_t *)q.keep_counts.p : nullptr));
  return pipe_finish(m, q, R, 1, scores, bboxes, keep_idx, keep_counts, ticket);
}

int mpn_model_detect_nms_submit(mpn_model *m, const float *image, int32_t H, int32_t W, const float *boxes, int64_t R,
                                float im_scale, float W0, float H0, float score_thresh, float nms_thr, float *scores,
                                float *bboxes, int32_t *keep_idx, int32_t *keep_counts, int32_t *ticket) {
  if (!m) return MPN_ERR_ARG;
  MPN_CHECK_ARG(m->ctx, image, "image missing");
  return submit_common(m, image, H, W, nullptr, 0, 0, nullptr, 0, 0, boxes, R, im_scale, W0, H0, score_thresh, nms_thr, scores, bboxes,
                       keep_idx, keep_counts, ticket);
}

int mpn_model_detect_nms_submit_u8(mpn_model *m, const uint8_t *im_hwc, int32_t H0, int32_t W0, const mpn_image_transform *tf,
                                   double scale, double max_size, const float *boxes, int64_t R, float score_thresh, float nms_thr,
                                   float *scores, float *bboxes, int32_t *keep_idx, int32_t *keep_counts, int32_t *ticket) {
  if (!m) return MPN_ERR_ARG;
  MPN_CHECK_ARG(m->ctx, im_hwc, "image missing");
  return submit_common(m, nullptr, 0, 0, im_hwc, H0, W0, tf, scale, max_size, boxes, R, 0.f, 0.f, 0.f, score_thresh, nms_thr, scores, bboxes,
                       keep_idx, keep_counts, ticket);
}

int mpn_model_detect_nms_batch_submit_u8(mpn_model *m, const uint8_t *ims_hwc, int32_t N, const int32_t *H0, const int32_t *W0,
                                         const mpn_image_transform *tf, double scale, double max_size, const float *boxes,
                                         const int64_t *img_offsets, float score_thresh, float nms_thr, float *scores, float *bboxes,
                                         int32_t *keep_idx, int32_t *keep_counts, int32_t *ticket) {
  if (!m) return MPN_ERR_ARG;
  mpn_ctx *ctx = m->ctx;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  // every check on the host, before anything is enqueued
  MPN_CHECK_ARG(ctx, N >= 1 && N <= MPN_MAX_BATCH, "batch size N must be in 1..MPN_MAX_BATCH");
  MPN_CHECK_ARG(ctx, ims_hwc && H0 && W0 && tf && boxes && img_offsets && ticket, "images / H0 / W0 / transformer / boxes / img_offsets / ticket missing");
  int32_t h[MPN_MAX_BATCH], w[MPN_MAX_BATCH], H = 0, W = 0; double s[MPN_MAX_BATCH]; size_t raw_bytes = 0;
  MPN_TRY(mpn_get_images_batch_check(ctx, N, H0, W0, tf, scale, max_size, h, w, s, H, W, raw_bytes));
  MPN_CHECK_ARG(ctx, H <= m->d.max_h && W <= m->d.max_w, "padded canvas larger than max_h x max_w");
  float sc[MPN_MAX_BATCH], w0[MPN_MAX_BATCH], h0[MPN_MAX_BATCH];
  for (int i = 0; i < N; ++i) { sc[i] = (float)s[i]; w0[i] = (float)W0[i]; h0[i] = (float)H0[i]; }   // as submit_common
  MpnBatch b; int cap = 0;
  MPN_TRY(batch_desc(m, N, img_offsets, sc, w0, h0, b, cap));
  MPN_CHECK_ARG(ctx, !m->sink || m->sink_n + N <= m->sink_cap, "detection sink is full (mpn_model_set_detection_sink capacity)");
  if (N == 1)        // one image: the single-image raw path, byte for byte
    return submit_common(m, nullptr, 0, 0, ims_hwc, H0[0], W0[0], tf, scale, max_size, boxes, img_offsets[1], 0.f, 0.f, 0.f, score_thresh,
                         nms_thr, scores, bboxes, keep_idx, keep_counts, ticket);
  mpn_model::PipeSlot *qp = nullptr;
  MPN_TRY(pipe_slot(m, qp));
  mpn_model::PipeSlot &q = *qp;
  const int C = m->d.num_classes;
  const int64_t R = b.off[N];
  MPN_TRY(q.image.ensure(ctx, sizeof(float) * 3 * (size_t)N * H * W));
  MPN_TRY(q.raw_u8.ensure(ctx, raw_bytes));
  MPN_TRY(q.boxes.ensure(ctx, sizeof(float) * 4 * (size_t)R));
  MPN_TRY(q.scores.ensure(ctx, sizeof(float) * (size_t)R * C));
  MPN_TRY(q.bboxes.ensure(ctx, sizeof(float) * (size_t)R * 4 * C));
  MPN_TRY(q.keep_idx.ensure(ctx, sizeof(int32_t) * (size_t)(C - 1) * R));
  MPN_TRY(q.keep_counts.ensure(ctx, sizeof(int32_t) * (size_t)N * (C - 1)));
  MPN_CUDA(ctx, cudaMemcpyAsync(q.raw_u8.p, ims_hwc, raw_bytes, cudaMemcpyHostToDevice, m->s_h2d));
  MPN_CUDA(ctx, cudaMemcpyAsync(q.boxes.p, boxes, sizeof(float) * 4 * (size_t)R, cudaMemcpyHostToDevice, m->s_h2d));
  MPN_CUDA(ctx, cudaEventRecord(q.h2d, m->s_h2d));
  MPN_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, q.h2d, 0));
  MPN_TRY(mpn_get_images_batch_launch(ctx, nullptr, (const uint8_t *)q.raw_u8.p, N, H0, W0, h, w, H, W, tf, (float *)q.image.p));
  MPN_TRY(detect_nms_batch_core(m, (const float *)q.image.p, N, H, W, (const float *)q.boxes.p, b, cap, score_thresh, nms_thr));
  MPN_TRY(detect_nms_batch_copy_out(m, b, cap, cudaMemcpyDeviceToDevice, scores ? (float *)q.scores.p : nullptr,
                                    bboxes ? (float *)q.bboxes.p : nullptr, keep_idx ? (int32_t *)q.keep_idx.p : nullptr,
                                    keep_counts ? (int32_t *)q.keep_counts.p : nullptr));
  return pipe_finish(m, q, R, N, scores, bboxes, keep_idx, keep_counts, ticket);
}

int mpn_model_detect_nms_wait(mpn_model *m, int32_t ticket) {
  if (!m) return MPN_ERR_ARG;
  mpn_ctx *ctx = m->ctx;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  mpn_model::PipeSlot &q = m->pipe[ticket & 1];
  MPN_CHECK_ARG(ctx, ticket >= 0 && q.busy && q.ticket == ticket, "unknown or already completed ticket");
  MPN_CUDA(ctx, cudaEventSynchronize(q.done));
  q.busy = false;
  return mpn_ovf_test(ctx);
}

// Tester_FRCNN:testOne (Tester_FRCNN.lua:54-139) entirely on the device: see include/mpn_abi.h
int mpn_model_test_one(mpn_model *m, const float *image, int32_t H, int32_t W, const float *boxes, int64_t R, float im_scale, float W0,
                       float H0, const mpn_test_opts *o, float *scores, float *bboxes, int32_t *keep_idx, int32_t *keep_counts, float *voted) {
  if (!m || !o) return MPN_ERR_ARG;
  mpn_ctx *ctx = m->ctx;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, image && boxes && R > 0, "image/boxes missing");
  MPN_CHECK_ARG(ctx, o->num_iter >= 1 && o->num_iter <= 8, "num_iter must be in 1..8");
  MPN_CHECK_ARG(ctx, !o->use_rbox_scores || o->num_iter > 1, "test_use_rbox_scores needs test_num_iterative_loc > 1 (Tester_FRCNN.lua:92)");
  MPN_CHECK_ARG(ctx, !o->bbox_voting || voted, "bbox voting needs the `voted` output");
  const int C = m->d.num_classes, n_it = o->num_iter;
  const int64_t n_out = R * (n_it - (o->use_rbox_scores ? 1 : 0));        // rows of the joined outputs
  MPN_CHECK_ARG(ctx, n_out < (1ll << 30), "too many rows");
  const size_t bs = sizeof(float) * (size_t)R * C, bb = sizeof(float) * (size_t)R * 4 * C;
  MPN_TRY(m->image_dev.ensure(ctx, sizeof(float) * 3 * (size_t)H * W));
  MPN_TRY(m->boxes_dev.ensure(ctx, sizeof(float) * 4 * (size_t)R));
  MPN_TRY(m->to_pass_scores.ensure(ctx, bs * n_it)); MPN_TRY(m->to_pass_bboxes.ensure(ctx, bb * n_it));
  MPN_TRY(m->to_new_boxes.ensure(ctx, sizeof(float) * 4 * (size_t)R));
  MPN_TRY(m->to_scores.ensure(ctx, sizeof(float) * (size_t)n_out * C)); MPN_TRY(m->to_bboxes.ensure(ctx, sizeof(float) * (size_t)n_out * 4 * C));
  MPN_TRY(m->to_sb.ensure(ctx, sizeof(float) * 5 * (size_t)(C - 1) * n_out)); MPN_TRY(m->to_src.ensure(ctx, sizeof(int32_t) * (size_t)(C - 1) * n_out));
  MPN_TRY(m->to_counts.ensure(ctx, sizeof(int32_t) * (size_t)C)); MPN_TRY(m->to_keep.ensure(ctx, sizeof(int32_t) * (size_t)(C - 1) * n_out));
  MPN_TRY(m->to_keep_counts.ensure(ctx, sizeof(int32_t) * (size_t)C));
  if (o->bbox_voting) MPN_TRY(m->to_voted.ensure(ctx, sizeof(float) * 5 * (size_t)(C - 1) * n_out));
  MPN_CUDA(ctx, cudaMemcpyAsync(m->image_dev.p, image, sizeof(float) * 3 * (size_t)H * W, cudaMemcpyHostToDevice, ctx->stream));
  MPN_CUDA(ctx, cudaMemcpyAsync(m->boxes_dev.p, boxes, sizeof(float) * 4 * (size_t)R, cudaMemcpyHostToDevice, ctx->stream));
  MPN_TRY(mpn_model_trunk_dev(m, (const float *)m->image_dev.p, H, W));
  auto ps = [&](int it) { return (float *)((char *)m->to_pass_scores.p + bs * it); };
  auto pb = [&](int it) { return (float *)((char *)m->to_pass_bboxes.p + bb * it); };
  // pass 1 on the proposals, clamped (:72-78); passes 2..n on nn.SelectBoxes of the previous pass, cached features, NOT clamped (:82-89)
  MPN_TRY(run_detect_pass(m, (const float *)m->boxes_dev.p, R, im_scale, 1, W0, H0, ps(0), pb(0)));
  for (int it = 1; it < n_it; ++it) {
    MPN_TRY(mpn_select_boxes_launch(ctx, ps(it - 1), pb(it - 1), R, C, nullptr, nullptr, (float *)m->to_new_boxes.p));
    MPN_TRY(run_detect_pass(m, (const float *)m->to_new_boxes.p, R, im_scale, 0, 0.f, 0.f, ps(it), pb(it)));
  }
  // joinTable (:99-100); with rbox scores the scores of pass i + 1 go with the boxes of pass i (:91-97)
  const int s0 = o->use_rbox_scores ? 1 : 0, n_blocks = n_it - s0;
  MPN_CUDA(ctx, cudaMemcpyAsync(m->to_scores.p, ps(s0), bs * n_blocks, cudaMemcpyDeviceToDevice, ctx->stream));
  MPN_CUDA(ctx, cudaMemcpyAsync(m->to_bboxes.p, pb(0), bb * n_blocks, cudaMemcpyDeviceToDevice, ctx->stream));
  MPN_TRY(mpn_gather_scored_launch(ctx, (const float *)m->to_scores.p, (const float *)m->to_bboxes.p, (int)n_out, C, o->score_thresh,
                                   (float *)m->to_sb.p, (int32_t *)m->to_src.p, (int32_t *)m->to_counts.p));
  MPN_TRY(mpn_nms_launch(ctx, (const float *)m->to_sb.p, (int)n_out, C - 1, (const int32_t *)m->to_counts.p, (const int32_t *)m->to_src.p,
                         o->nms_thr, (int32_t *)m->to_keep.p, (int32_t *)m->to_keep_counts.p));
  if (o->bbox_voting)
    MPN_TRY(mpn_bbox_vote_batched_launch(ctx, (const float *)m->to_sb.p, (const int32_t *)m->to_counts.p, (const int32_t *)m->to_keep.p,
                                         (const int32_t *)m->to_keep_counts.p, (const float *)m->to_scores.p, (const float *)m->to_bboxes.p, C,
                                         (int)n_out, o->vote_thr, o->vote_score_pow, (float *)m->to_voted.p));
  if (scores) MPN_CUDA(ctx, cudaMemcpyAsync(scores, m->to_scores.p, sizeof(float) * (size_t)n_out * C, cudaMemcpyDeviceToHost, ctx->stream));
  if (bboxes) MPN_CUDA(ctx, cudaMemcpyAsync(bboxes, m->to_bboxes.p, sizeof(float) * (size_t)n_out * 4 * C, cudaMemcpyDeviceToHost, ctx->stream));
  if (keep_idx) MPN_CUDA(ctx, cudaMemcpyAsync(keep_idx, m->to_keep.p, sizeof(int32_t) * (size_t)(C - 1) * n_out, cudaMemcpyDeviceToHost, ctx->stream));
  if (keep_counts) MPN_CUDA(ctx, cudaMemcpyAsync(keep_counts, m->to_keep_counts.p, sizeof(int32_t) * (size_t)(C - 1), cudaMemcpyDeviceToHost, ctx->stream));
  if (voted && o->bbox_voting) MPN_CUDA(ctx, cudaMemcpyAsync(voted, m->to_voted.p, sizeof(float) * 5 * (size_t)(C - 1) * n_out, cudaMemcpyDeviceToHost, ctx->stream));
  MPN_TRY(mpn_ovf_copy_async(ctx, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return mpn_ovf_test(ctx);
}

int mpn_model_set_detection_sink(mpn_model *m, float *records_dev, int64_t capacity, int32_t top_k) {
  if (!m) return MPN_ERR_ARG;
  mpn_ctx *ctx = m->ctx;
  MPN_CHECK_ARG(ctx, !records_dev || (capacity > 0 && top_k >= 1 && top_k <= MPN_MAX_DET), "detection sink: capacity > 0 and 1 <= top_k <= MPN_MAX_DET");
  m->sink = records_dev; m->sink_cap = records_dev ? capacity : 0; m->sink_n = 0; m->sink_top_k = records_dev ? top_k : 100;
  return MPN_OK;
}

int mpn_model_detection_sink_count(const mpn_model *m, int64_t *n_records) {
  if (!m || !n_records) return MPN_ERR_ARG;
  *n_records = m->sink_n;
  return MPN_OK;
}

int mpn_model_get_pooled(mpn_model *m, int32_t tower, int64_t r0, int64_t n, float *out, int64_t capacity, int64_t *R_total,
                         int32_t *bins, int32_t *Ctot) {
  if (!m) return MPN_ERR_ARG;
  mpn_ctx *ctx = m->ctx;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, m->heads_planned && tower >= 0 && tower < (int)m->tex.size(), "no heads pass yet, or unknown tower");
  const DTensor &t = m->tex[tower].pooled;
  const int64_t row = t.H * t.W * t.C;
  if (R_total) *R_total = t.N;
  if (bins) *bins = (int32_t)(t.H * t.W);
  if (Ctot) *Ctot = (int32_t)t.C;
  if (!out) return MPN_OK;
  MPN_CHECK_ARG(ctx, r0 >= 0 && n > 0 && r0 + n <= t.N && capacity >= n * row, "row range outside the pooled tensor, or buffer too small");
  void *tmp = nullptr;
  MPN_TRY(mpn_scratch(ctx, sizeof(float) * (size_t)(n * row), &tmp));
  MPN_TRY(mpn_join_rows_launch(ctx, t.hi + r0 * row, t.lo + r0 * row, n, row, row, t.fmt, (float *)tmp));
  MPN_CUDA(ctx, cudaMemcpyAsync(out, tmp, sizeof(float) * (size_t)(n * row), cudaMemcpyDeviceToHost, ctx->stream));
  MPN_TRY(mpn_ovf_copy_async(ctx, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return mpn_ovf_test(ctx);
}

int mpn_model_get_trunk_slot(mpn_model *m, int32_t slot, float *out_nchw, int64_t capacity, int32_t *C, int32_t *H,
                             int32_t *W) {
  if (!m) return MPN_ERR_ARG;
  mpn_ctx *ctx = m->ctx;
  MPN_CUDA(ctx, cudaSetDevice(ctx->device));
  MPN_CHECK_ARG(ctx, m->trunk_valid && slot > 0 && m->trunk_slots.count(slot), "unknown trunk slot or no trunk forward yet");
  MPN_CHECK_ARG(ctx, !m->elided_slots.count(slot),
                "trunk slot was fused into the following max pool and never written (mpn_model_set_conv_impl(m, 2) disables the fusion)");
  const DTensor &t = m->trunk_slots[slot];
  const int64_t n = t.N * t.C * t.H * t.W;
  if (C) *C = (int32_t)t.C; if (H) *H = (int32_t)t.H; if (W) *W = (int32_t)t.W;
  if (!out_nchw) return MPN_OK;
  MPN_CHECK_ARG(ctx, capacity >= n, "output buffer too small");
  void *tmp = nullptr;
  MPN_TRY(mpn_scratch(ctx, sizeof(float) * (size_t)n, &tmp));
  MPN_TRY(mpn_nhwc_split_to_nchw_launch(ctx, t, (float *)tmp));
  MPN_CUDA(ctx, cudaMemcpyAsync(out_nchw, tmp, sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
  MPN_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MPN_OK;
}

}  // extern "C"
