// Whole-model extractor for the TDNN x-vector family: frame-level TDNN layers -> statistics
// pooling -> segment-level affine layers.  Owns packed weights and workspace on the current device.
// Stands in for Xvector.extract_embedding (pytorch/model/xvector.py:77-98) on a whole batch of
// equal-length utterances and for the "load weights, run extraction without Python" role of the
// reference's C++ runtime (runtime/bin/extractor_main.cc, runtime/speaker/torch_asv_model.cc).
#include <cuda_runtime.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <numeric>
#include <tuple>
#include <utility>
#include <vector>

#include "common.cuh"

namespace xvb {

struct Layer {
  int Cin = 0, Cout = 0, ntaps = 0, flags = 0;
  int ctx[XVB_MAX_TAPS] = {0};
  uint16_t* w_hi = nullptr;
  uint16_t* w_lo = nullptr;
  float* bias = nullptr;
  float* scale = nullptr;
  float* shift = nullptr;
};

template <typename T>
static int dev_alloc(T** p, size_t n) {
  XVB_CUDA(cudaMalloc((void**)p, n * sizeof(T)));
  return XVB_OK;
}

// Everything one (B, T) batch shape needs besides launches: a GemmPlan per layer (tensor maps over the
// extractor's own workspace, tile geometry, kernel instantiation) and the split-K scratch those plans own.
struct StepPlan {
  std::vector<GemmPlan*> frame, segment;
  std::vector<void*> scratch;
  int pool_blocks = 0, pool_tb = 0;
  ~StepPlan() {
    for (GemmPlan* g : frame) gemm_plan_destroy(g);
    for (GemmPlan* g : segment) gemm_plan_destroy(g);
    for (void* q : scratch) cudaFree(q);
  }
};

}  // namespace xvb

using namespace xvb;

struct xvb_extractor {
  int feat_dim = 0, ldf = 0;
  bool finalized = false;
  float pooling_eps = 1e-10f;
  std::vector<Layer> frame, segment;
  // workspace
  long long cap_frames = 0;
  int cap_B = 0;
  uint16_t* in_hi = nullptr; uint16_t* in_lo = nullptr;        // (B,T,ldf)
  uint16_t* act_hi[2] = {nullptr, nullptr};                    // ping-pong (B,T,max_c)
  uint16_t* act_lo[2] = {nullptr, nullptr};
  float* last_f32 = nullptr;                                   // (B,T,C_last)
  float* stats = nullptr;                                      // (B,2*C_last)
  float* emb_ws = nullptr;                                     // (B,D): nominal target of the last layer's plan
  uint16_t* stats_hi = nullptr; uint16_t* stats_lo = nullptr;
  uint16_t* seg_hi[2] = {nullptr, nullptr}; uint16_t* seg_lo[2] = {nullptr, nullptr};  // (B,max_seg_c)
  float* h_feats = nullptr; float* h_emb = nullptr;            // device staging for *_host
  size_t h_feats_cap = 0, h_emb_cap = 0;
  // double-buffered pipelined host path (submit/wait): H2D of batch i+1 overlaps the stack of batch i
  // (slots 0/1 serve submit_host/wait; the shard call uses all kSlots: two per lane, so a lane's next batch is already
  // on the device when its current one finishes)
  static constexpr int kSlots = 4;
  float* p_feats[kSlots] = {nullptr, nullptr, nullptr, nullptr}; float* p_emb[kSlots] = {nullptr, nullptr, nullptr, nullptr};
  size_t p_feats_cap[kSlots] = {0, 0, 0, 0}, p_emb_cap[kSlots] = {0, 0, 0, 0};
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_h2d[kSlots] = {nullptr, nullptr, nullptr, nullptr}, ev_done[kSlots] = {nullptr, nullptr, nullptr, nullptr};
  bool slot_busy[2] = {false, false};
  int max_c = 0, max_seg_c = 0;
  int last_launches = 0;
  // optional per-kernel CUDA-event timing on the launching stream (bench.py roofline)
  bool fused_pooling = true;
  // first layer as an im2col view (consecutive context taps over a time-padded frame matrix): 7 channel
  // blocks instead of 10 for [-2..2] x 80.  Turned off if the driver rejects the overlapping tensor map.
  bool im2col_first = false;
  int pad_front = 0, pad_back = 0;
  float* pool_partial = nullptr;
  size_t pool_partial_cap = 0;
  // ragged batches: [offsets (B+1) | lengths (B)] of the current batch on the device (2 * cap_B + 1 int32, part of the
  // workspace), its pinned host staging and the event that tells when the last upload has left the staging buffer
  int32_t* ragged_meta = nullptr;
  int32_t* ragged_meta_host = nullptr;
  size_t ragged_meta_host_cap = 0;
  cudaEvent_t ev_meta = nullptr;
  float* ragged_emb_host = nullptr;          // shard call: embeddings in batch (length-sorted) order, pinned
  size_t ragged_emb_host_cap = 0;
  int32_t* shard_meta = nullptr;             // shard call: every batch's [offsets | lengths] block
  size_t shard_meta_cap = 0;
  // launch plans per batch shape (B, T, ragged); they hold pointers into the workspace, so anything that reallocates it
  // clears them.  Every plan owns split-K scratch, and a stream of ragged batches can visit many padded lengths, so
  // the ragged plans are dropped together once there are kMaxRaggedPlans of them.
  static constexpr int kMaxRaggedPlans = 64;
  std::map<std::tuple<int, int, bool>, StepPlan*> plans;
  int ragged_plans = 0;
  void drop_plans() {
    for (auto& kv : plans) delete kv.second;
    plans.clear();
    ragged_plans = 0;
  }
  void drop_ragged_plans() {
    for (auto it = plans.begin(); it != plans.end();) {
      if (std::get<2>(it->first)) { delete it->second; it = plans.erase(it); }
      else ++it;
    }
    ragged_plans = 0;
  }
  // Two-lane shard pipeline: batches of a shard alternate between this extractor and `lane1`, a shallow twin that
  // shares the packed weights but owns its workspace and plans, each on its own stream.  The tcgen05 layer kernels
  // occupy whole SMs, so the two lanes' GEMMs queue behind one another; what overlaps is everything else -- the
  // bandwidth-bound staging / pooling-merge / split-K-reduce kernels of one batch run on the SMs' spare thread and
  // register slots next to the other batch's GEMM CTAs, and a GEMM's ragged tail is filled by the other lane's CTAs.
  xvb_extractor* lane1 = nullptr;
  bool is_lane = false;                      // a twin does not own the weights
  // replicated embedding table (peer.cu): every batch's rows go to all these copies as soon as they exist
  float* gather_tables[XVB_MAX_PEERS] = {nullptr};
  int gather_n = 0;
  int64_t gather_row0 = 0, gather_ld = 0;
  cudaStream_t lane_stream[2] = {nullptr, nullptr};
  cudaEvent_t ev_lane_start = nullptr, ev_lane_done[2] = {nullptr, nullptr};
  bool profiling = false;
  bool in_shard = false;
  std::vector<cudaEvent_t> events;
  int events_used = 0;
  cudaStream_t events_stream = nullptr;

  int mark(cudaStream_t s) {
    if (!profiling) return XVB_OK;
    if (events_used == (int)events.size()) {
      cudaEvent_t e;
      XVB_CUDA(cudaEventCreate(&e));
      events.push_back(e);
    }
    XVB_CUDA(cudaEventRecord(events[events_used++], s));
    return XVB_OK;
  }

  void free_ws() {
    drop_plans();
    cudaFree(in_hi); cudaFree(in_lo);
    for (int i = 0; i < 2; ++i) { cudaFree(act_hi[i]); cudaFree(act_lo[i]); cudaFree(seg_hi[i]); cudaFree(seg_lo[i]); }
    cudaFree(last_f32); cudaFree(stats); cudaFree(stats_hi); cudaFree(stats_lo); cudaFree(emb_ws); cudaFree(ragged_meta);
    in_hi = in_lo = nullptr; last_f32 = stats = emb_ws = nullptr; stats_hi = stats_lo = nullptr; ragged_meta = nullptr;
    for (int i = 0; i < 2; ++i) act_hi[i] = act_lo[i] = seg_hi[i] = seg_lo[i] = nullptr;
    cap_frames = 0; cap_B = 0;
  }
};

static int upload_layer(Layer& L, int Cin, int Cout, const int* ctx, int ntaps, const float* w_host,
                        const float* bias_host, const float* scale_host, const float* shift_host, int flags) {
  XVB_CHECK_ARG(ntaps >= 1 && ntaps <= XVB_MAX_TAPS && ctx && w_host, "add layer: bad taps/weights");
  XVB_CHECK_ARG(!(flags & XVB_BN) || (scale_host && shift_host), "add layer: XVB_BN without scale/shift");
  for (int i = 1; i < ntaps; ++i) XVB_CHECK_ARG(ctx[i] > ctx[i - 1], "add layer: context must be strictly increasing");
  // left/right/total context exactly as TdnnAffine.__init__ (components.py:50-53)
  const int left = ctx[0] < 0 ? ctx[0] : 0;
  const int right = ctx[ntaps - 1] > 0 ? ctx[ntaps - 1] : 0;
  const int tot = right - left + 1;
  L.Cin = Cin; L.Cout = Cout; L.ntaps = ntaps; L.flags = flags;
  for (int i = 0; i < ntaps; ++i) L.ctx[i] = ctx[i];
  const size_t wn = (size_t)Cout * Cin * tot;
  float* w_dev = nullptr;
  int rc = dev_alloc(&w_dev, wn);
  if (rc) return rc;
  XVB_CUDA(cudaMemcpy(w_dev, w_host, wn * sizeof(float), cudaMemcpyHostToDevice));
  const size_t pn = (size_t)xvb_packed_weight_elems(Cout, Cin, ntaps);
  if ((rc = dev_alloc(&L.w_hi, pn))) return rc;
  if ((rc = dev_alloc(&L.w_lo, pn))) return rc;
  rc = xvb_pack_tdnn_weight(w_dev, Cout, Cin, tot, left, ctx, ntaps, L.w_hi, L.w_lo, nullptr);
  if (rc) return rc;
  XVB_CUDA(cudaDeviceSynchronize());
  cudaFree(w_dev);
  auto up = [&](float** d, const float* h) -> int {
    if (!h) return XVB_OK;
    int r = dev_alloc(d, (size_t)Cout);
    if (r) return r;
    XVB_CUDA(cudaMemcpy(*d, h, (size_t)Cout * sizeof(float), cudaMemcpyHostToDevice));
    return XVB_OK;
  };
  if ((rc = up(&L.bias, bias_host))) return rc;
  if (flags & XVB_BN) {
    if ((rc = up(&L.scale, scale_host))) return rc;
    if ((rc = up(&L.shift, shift_host))) return rc;
  }
  return XVB_OK;
}

extern "C" int xvb_extractor_create(xvb_extractor_t** out, int feat_dim) {
  int rc = require_sm100();
  if (rc) return rc;
  XVB_CHECK_ARG(out && feat_dim > 0, "xvb_extractor_create: bad arguments");
  xvb_extractor* h = new xvb_extractor();
  h->feat_dim = feat_dim;
  h->ldf = (int)round_up(feat_dim, 8);
  *out = h;
  return XVB_OK;
}

extern "C" int xvb_extractor_add_frame_layer(xvb_extractor_t* h, int Cout, const int* context_host, int ntaps,
                                             const float* w_host, const float* bias_host, const float* bn_scale_host,
                                             const float* bn_shift_host, int flags) {
  XVB_CHECK_ARG(h && !h->finalized, "xvb_extractor_add_frame_layer: null or finalized extractor");
  XVB_CHECK_ARG(h->segment.empty(), "xvb_extractor_add_frame_layer: frame layers must precede segment layers");
  const int Cin = h->frame.empty() ? h->feat_dim : h->frame.back().Cout;
  Layer L;
  int rc = upload_layer(L, Cin, Cout, context_host, ntaps, w_host, bias_host, bn_scale_host, bn_shift_host, flags);
  if (rc) return rc;
  h->frame.push_back(L);
  return XVB_OK;
}

extern "C" int xvb_extractor_add_segment_layer(xvb_extractor_t* h, int Cout, const float* w_host, const float* bias_host,
                                               const float* bn_scale_host, const float* bn_shift_host, int flags) {
  XVB_CHECK_ARG(h && !h->finalized && !h->frame.empty(), "xvb_extractor_add_segment_layer: need frame layers first");
  const int Cin = h->segment.empty() ? 2 * h->frame.back().Cout : h->segment.back().Cout;
  const int ctx0 = 0;
  Layer L;
  int rc = upload_layer(L, Cin, Cout, &ctx0, 1, w_host, bias_host, bn_scale_host, bn_shift_host, flags);
  if (rc) return rc;
  h->segment.push_back(L);
  return XVB_OK;
}

extern "C" int xvb_extractor_finalize(xvb_extractor_t* h, float pooling_eps) {
  XVB_CHECK_ARG(h && !h->frame.empty() && !h->segment.empty(), "xvb_extractor_finalize: need >=1 frame and >=1 segment layer");
  h->max_c = 0;
  for (size_t i = 0; i + 1 < h->frame.size(); ++i) {
    XVB_CHECK_ARG(h->frame[i].Cout % 8 == 0, "frame layer %d: Cout=%d must be a multiple of 8", (int)i, h->frame[i].Cout);
    if (h->frame[i].Cout > h->max_c) h->max_c = h->frame[i].Cout;
  }
  XVB_CHECK_ARG(h->frame.back().Cout % 4 == 0, "last frame layer: Cout=%d must be a multiple of 4", h->frame.back().Cout);
  h->max_seg_c = 0;
  for (size_t i = 0; i + 1 < h->segment.size(); ++i) {
    XVB_CHECK_ARG(h->segment[i].Cout % 8 == 0, "segment layer %d: Cout must be a multiple of 8", (int)i);
    if (h->segment[i].Cout > h->max_seg_c) h->max_seg_c = h->segment[i].Cout;
  }
  XVB_CHECK_ARG(h->segment.back().Cout % 4 == 0, "last segment layer: Cout must be a multiple of 4");
  h->pooling_eps = pooling_eps;
  {
    const Layer& L0 = h->frame[0];
    bool consecutive = L0.ntaps > 1 && L0.ctx[0] <= 0 && L0.ctx[L0.ntaps - 1] >= 0;
    for (int i = 1; i < L0.ntaps; ++i) consecutive = consecutive && L0.ctx[i] == L0.ctx[i - 1] + 1;
    const int knob = getenv("XVB_IM2COL") ? atoi(getenv("XVB_IM2COL")) : 1;   // read per extractor: tests flip it
    h->im2col_first = knob && consecutive && h->feat_dim % 16 == 0;   // plane pitch == packed tap pitch
    h->pad_front = h->im2col_first ? -L0.ctx[0] : 0;
    h->pad_back = h->im2col_first ? L0.ctx[L0.ntaps - 1] : 0;
  }
  h->finalized = true;
  return XVB_OK;
}

extern "C" int xvb_extractor_embed_dim(const xvb_extractor_t* h) {
  return (h && !h->segment.empty()) ? h->segment.back().Cout : XVB_ESTATE;
}

static int reserve(xvb_extractor* h, int B, int T) {
  const long long frames = (long long)B * T;
  if (frames <= h->cap_frames && B <= h->cap_B) return XVB_OK;
  const long long nf = frames > h->cap_frames ? frames : h->cap_frames;
  const int nb = B > h->cap_B ? B : h->cap_B;
  h->free_ws();
  int rc;
  const size_t in_rows = (size_t)nf + (size_t)nb * (h->pad_front + h->pad_back);
  if ((rc = dev_alloc(&h->in_hi, in_rows * h->ldf))) return rc;
  if ((rc = dev_alloc(&h->in_lo, in_rows * h->ldf))) return rc;
  if (h->max_c > 0)
    for (int i = 0; i < 2; ++i) {
      if ((rc = dev_alloc(&h->act_hi[i], (size_t)nf * h->max_c))) return rc;
      if ((rc = dev_alloc(&h->act_lo[i], (size_t)nf * h->max_c))) return rc;
    }
  const int cl = h->frame.back().Cout;
  if ((rc = dev_alloc(&h->last_f32, (size_t)nf * cl))) return rc;
  if ((rc = dev_alloc(&h->stats, (size_t)nb * 2 * cl))) return rc;
  if ((rc = dev_alloc(&h->emb_ws, (size_t)nb * h->segment.back().Cout))) return rc;
  if ((rc = dev_alloc(&h->stats_hi, (size_t)nb * 2 * cl))) return rc;
  if ((rc = dev_alloc(&h->stats_lo, (size_t)nb * 2 * cl))) return rc;
  if (h->max_seg_c > 0)
    for (int i = 0; i < 2; ++i) {
      if ((rc = dev_alloc(&h->seg_hi[i], (size_t)nb * h->max_seg_c))) return rc;
      if ((rc = dev_alloc(&h->seg_lo[i], (size_t)nb * h->max_seg_c))) return rc;
    }
  if ((rc = dev_alloc(&h->ragged_meta, (size_t)2 * nb + 1))) return rc;
  h->cap_frames = nf;
  h->cap_B = nb;
  return XVB_OK;
}

// Build the launch plan of one batch shape (see StepPlan).  On failure nothing is cached.  A ragged plan's frame layers
// mask with the lengths of the batch's [offsets | lengths] block in h->ragged_meta.
static int build_step_plan(xvb_extractor* h, int B, int T, bool ragged, StepPlan** out) {
  StepPlan* sp = new StepPlan();
  struct Guard { StepPlan* p; ~Guard() { delete p; } } guard{sp};
  int rc;
  sp->pool_blocks = xvb_pool_partial_blocks(B, T, &sp->pool_tb);
  const uint16_t* x_hi = h->in_hi;
  const uint16_t* x_lo = h->in_lo;
  int64_t ldx = h->ldf;
  auto add = [&](std::vector<GemmPlan*>& dst, const xvb_tdnn_args_t& a) -> int {
    void* scratch = nullptr;
    const size_t need = gemm_plan_scratch_bytes(a);
    if (need) {
      XVB_CUDA(cudaMalloc(&scratch, need));
      sp->scratch.push_back(scratch);
    }
    GemmPlan* g = nullptr;
    int r = gemm_plan_build(&g, a, nullptr, scratch);
    if (r) return r;
    dst.push_back(g);
    return XVB_OK;
  };
  for (size_t i = 0; i < h->frame.size(); ++i) {
    const Layer& L = h->frame[i];
    const bool last = i + 1 == h->frame.size();
    uint16_t* y_hi = last ? nullptr : h->act_hi[i & 1];
    uint16_t* y_lo = last ? nullptr : h->act_lo[i & 1];
    xvb_tdnn_args_t a{};
    a.x_hi = x_hi; a.x_lo = x_lo; a.ldx = ldx; a.w_hi = L.w_hi; a.w_lo = L.w_lo;
    a.bias = L.bias; a.bn_scale = L.scale; a.bn_shift = L.shift; a.flags = L.flags;
    a.context_host = L.ctx; a.ntaps = L.ntaps;
    a.y_hi = y_hi; a.y_lo = y_lo; a.ldy = L.Cout;
    a.B = B; a.T = T; a.Cin = L.Cin; a.Cout = L.Cout;
    if (ragged) a.lengths = h->ragged_meta + B + 1;
    const int ctx0 = 0;
    if (i == 0 && h->im2col_first) {   // window of ntaps consecutive frames = one long row of the padded planes
      a.context_host = &ctx0; a.ntaps = 1; a.Cin = L.ntaps * L.Cin;
      a.x_batch_stride = (int64_t)(T + h->pad_front + h->pad_back) * ldx;
    }
    if (last && h->fused_pooling) {
      a.pool_partial = h->pool_partial;
    } else if (last) {
      a.y_f32 = h->last_f32; a.ldyf = L.Cout;
    }
    rc = add(sp->frame, a);
    if (rc && i == 0 && h->im2col_first) return -1000;   // overlapping tensor map refused: caller falls back for good
    if (rc) return rc;
    x_hi = y_hi; x_lo = y_lo; ldx = L.Cout;
  }
  const int cl = h->frame.back().Cout;
  x_hi = h->stats_hi; x_lo = h->stats_lo; ldx = 2 * cl;
  for (size_t i = 0; i < h->segment.size(); ++i) {
    const Layer& L = h->segment[i];
    const bool last = i + 1 == h->segment.size();
    uint16_t* y_hi = last ? nullptr : h->seg_hi[i & 1];
    uint16_t* y_lo = last ? nullptr : h->seg_lo[i & 1];
    xvb_tdnn_args_t a{};
    a.x_hi = x_hi; a.x_lo = x_lo; a.ldx = ldx; a.w_hi = L.w_hi; a.w_lo = L.w_lo;
    a.bias = L.bias; a.bn_scale = L.scale; a.bn_shift = L.shift; a.flags = L.flags;
    a.context_host = L.ctx; a.ntaps = 1;
    a.y_hi = y_hi; a.y_lo = y_lo; a.ldy = L.Cout;
    if (last) { a.y_f32 = h->emb_ws; a.ldyf = L.Cout; }   // redirected to the caller's matrix at launch
    a.B = B; a.T = 1; a.Cin = L.Cin; a.Cout = L.Cout;
    if ((rc = add(sp->segment, a))) return rc;
    x_hi = y_hi; x_lo = y_lo; ldx = L.Cout;
  }
  guard.p = nullptr;
  *out = sp;
  return XVB_OK;
}

// The whole stack for one batch.  Equal lengths: feats (B, T, F).  Ragged (`ragged`): feats (sum_T, F) laid out by the
// offsets already in h->ragged_meta, T = the padded length Tq.
static int run_stack(xvb_extractor* h, const float* feats, int B, int T, bool ragged, float* emb, void* stream) {
  int rc = reserve(h, B, T);
  if (rc) return rc;
  const long before = g_launches;
  cudaStream_t cs = (cudaStream_t)stream;
  if (!h->in_shard) h->events_used = 0;   // a shard call keeps the events of all its batches
  h->events_stream = cs;
  StepPlan* sp = nullptr;
  const auto key = std::make_tuple(B, T, ragged);
  auto it = h->plans.find(key);
  if (it != h->plans.end()) {
    sp = it->second;
  } else {
    if (h->fused_pooling) {   // partials of the fused pooling epilogue: (time blocks, B, 2C) fp32
      int tb = 0;
      const size_t need = (size_t)xvb_pool_partial_blocks(B, T, &tb) * B * 2 * h->frame.back().Cout;
      if (need > h->pool_partial_cap) {
        h->drop_plans();      // they point into the old buffer
        cudaFree(h->pool_partial);
        h->pool_partial = nullptr; h->pool_partial_cap = 0;
        if ((rc = dev_alloc(&h->pool_partial, need))) return rc;
        h->pool_partial_cap = need;
      }
    }
    if (ragged && h->ragged_plans >= xvb_extractor::kMaxRaggedPlans) h->drop_ragged_plans();
    rc = build_step_plan(h, B, T, ragged, &sp);
    if (rc == -1000) {        // the driver refused the overlapping (im2col) tensor map: plain first layer from now on
      h->im2col_first = false;
      h->pad_front = h->pad_back = 0;
      h->drop_plans();
      return run_stack(h, feats, B, T, ragged, emb, stream);
    }
    if (rc) return rc;
    h->plans[key] = sp;
    if (ragged) ++h->ragged_plans;
  }
  if ((rc = h->mark(cs))) return rc;
  // 1. stage the frame matrix as split planes (framework.py:28-33 staging); for the im2col first layer with
  //    the zero frames of F.pad (components.py:117) written out around every utterance
  if (ragged)   // zero frames from L_b on: what the reference's per-utterance F.pad reads past the end
    rc = split_ragged_frames(feats, h->ragged_meta, B, T, h->feat_dim, h->in_hi, h->in_lo, h->ldf, h->pad_front, h->pad_back,
                             stream);
  else if (h->im2col_first)
    rc = xvb_split_frames(feats, B, T, h->feat_dim, h->in_hi, h->in_lo, h->ldf, h->pad_front, h->pad_back, stream);
  else
    rc = xvb_split_f32(feats, (int64_t)B * T, h->feat_dim, h->feat_dim, h->in_hi, h->in_lo, h->ldf, stream);
  if (rc) return rc;
  if ((rc = h->mark(cs))) return rc;
  // 2. frame-level TDNN stack (xvector.py:85-89)
  for (GemmPlan* g : sp->frame) {
    if ((rc = gemm_plan_launch(g, stream))) return rc;
    if ((rc = h->mark(cs))) return rc;
  }
  // 3. statistics pooling (xvector.py:90, pooling.py:58-67)
  const int cl = h->frame.back().Cout;
  if (h->fused_pooling)   // ragged: mean and std over each utterance's own L_b frames
    rc = pool_finalize_launch(h->pool_partial, sp->pool_blocks, sp->pool_tb, B, T, cl, h->pooling_eps, 0,
                              ragged ? h->ragged_meta + B + 1 : nullptr, h->stats, h->stats_hi, h->stats_lo, 2 * cl, stream);
  else
    rc = xvb_stats_pool(h->last_f32, cl, B, T, cl, h->pooling_eps, h->stats, h->stats_hi, h->stats_lo, 2 * cl, stream);
  if (rc) return rc;
  if ((rc = h->mark(cs))) return rc;
  // 4. segment-level layers (xvector.py:92-96); the last one writes the caller's embedding matrix
  for (size_t i = 0; i < sp->segment.size(); ++i) {
    const bool last = i + 1 == sp->segment.size();
    if ((rc = gemm_plan_launch(sp->segment[i], stream, last ? emb : nullptr))) return rc;
    if ((rc = h->mark(cs))) return rc;
  }
  h->last_launches = (int)(g_launches - before);
  return XVB_OK;
}

extern "C" int xvb_extractor_extract(xvb_extractor_t* h, const float* feats, int B, int T, float* emb, void* stream) {
  XVB_CHECK_ARG(h && h->finalized, "xvb_extractor_extract: extractor not finalized");
  XVB_CHECK_ARG(feats && emb && B > 0 && T > 0, "xvb_extractor_extract: bad arguments");
  return run_stack(h, feats, B, T, false, emb, stream);
}

static constexpr int kRaggedQuantum = 32;                 // padded length Tq = round_up(max L_b, 32)
static constexpr int64_t kRaggedDefaultMaxFrames = 262144;  // 256 utterances x 1024 frames

// The ragged path needs the fused pooling epilogue (the only pooling that counts per-utterance lengths) and writes no
// replicated table.
static int ragged_state_ok(const xvb_extractor* h, const char* fn) {
  if (!h->fused_pooling) { set_error("%s: needs fused pooling (xvb_extractor_set_fused_pooling(h, 1))", fn); return XVB_ESTATE; }
  if (h->gather_n) { set_error("%s: a gather table is set; ragged batches do not write replicated tables", fn); return XVB_ESTATE; }
  return XVB_OK;
}

extern "C" int xvb_extractor_extract_ragged(xvb_extractor_t* h, const float* feats, const int32_t* offsets_host, int B, float* emb,
                                            void* stream) {
  XVB_CHECK_ARG(h && h->finalized, "xvb_extractor_extract_ragged: extractor not finalized");
  XVB_CHECK_ARG(feats && offsets_host && emb && B > 0 && offsets_host[0] >= 0, "xvb_extractor_extract_ragged: bad arguments");
  int rc = ragged_state_ok(h, "xvb_extractor_extract_ragged");
  if (rc) return rc;
  int max_len = 0;
  for (int b = 0; b < B; ++b) {
    const int len = offsets_host[b + 1] - offsets_host[b];
    XVB_CHECK_ARG(offsets_host[b + 1] > offsets_host[b], "xvb_extractor_extract_ragged: utterance %d has %d frames (need >= 1)", b, len);
    max_len = len > max_len ? len : max_len;
  }
  XVB_CHECK_ARG(max_len <= (1 << 30), "xvb_extractor_extract_ragged: utterance too long");
  const int Tq = (int)round_up(max_len, kRaggedQuantum);
  if ((rc = reserve(h, B, Tq))) return rc;   // before the upload: it may reallocate ragged_meta
  cudaStream_t s = (cudaStream_t)stream;
  const size_t n = (size_t)2 * B + 1;
  if (!h->ev_meta) XVB_CUDA(cudaEventCreateWithFlags(&h->ev_meta, cudaEventDisableTiming));
  XVB_CUDA(cudaEventSynchronize(h->ev_meta));   // the previous upload has left the pinned staging buffer
  if (n > h->ragged_meta_host_cap) {
    cudaFreeHost(h->ragged_meta_host);
    h->ragged_meta_host = nullptr; h->ragged_meta_host_cap = 0;
    XVB_CUDA(cudaMallocHost((void**)&h->ragged_meta_host, n * sizeof(int32_t)));
    h->ragged_meta_host_cap = n;
  }
  for (int b = 0; b <= B; ++b) h->ragged_meta_host[b] = offsets_host[b];
  for (int b = 0; b < B; ++b) h->ragged_meta_host[B + 1 + b] = offsets_host[b + 1] - offsets_host[b];
  // on the launching stream: the kernels of an earlier batch on it have read the old block before this overwrites it
  XVB_CUDA(cudaMemcpyAsync(h->ragged_meta, h->ragged_meta_host, n * sizeof(int32_t), cudaMemcpyHostToDevice, s));
  XVB_CUDA(cudaEventRecord(h->ev_meta, s));
  return run_stack(h, feats, B, Tq, true, emb, stream);
}

extern "C" int xvb_ragged_plan(const int64_t* offsets_host, int64_t N, int batch, int64_t max_frames, int32_t* order_out,
                               int64_t* batch_first_out, int64_t* num_batches_out) {
  XVB_CHECK_ARG(offsets_host && order_out && batch_first_out && num_batches_out && N > 0 && N <= INT32_MAX && batch > 0 &&
                offsets_host[0] >= 0, "xvb_ragged_plan: bad arguments");
  if (max_frames <= 0) max_frames = kRaggedDefaultMaxFrames;
  for (int64_t i = 0; i < N; ++i) {
    const int64_t len = offsets_host[i + 1] - offsets_host[i];
    XVB_CHECK_ARG(len >= 1 && len <= (1 << 30), "xvb_ragged_plan: utterance %lld has %lld frames (need 1 .. 2^30)", (long long)i,
                  (long long)len);
  }
  auto len = [&](int32_t i) { return offsets_host[i + 1] - offsets_host[i]; };
  std::iota(order_out, order_out + N, 0);
  std::stable_sort(order_out, order_out + N, [&](int32_t a, int32_t b) { return len(a) < len(b); });
  // ascending lengths: the utterance that joins a batch sets its padded length
  int64_t nb = 0;
  for (int64_t i = 0; i < N;) {
    batch_first_out[nb++] = i;
    int64_t j = i + 1;
    while (j < N && j - i < batch && (j - i + 1) * round_up(len(order_out[j]), kRaggedQuantum) <= max_frames) ++j;
    i = j;
  }
  batch_first_out[nb] = N;
  *num_batches_out = nb;
  return XVB_OK;
}

extern "C" int xvb_extractor_set_gather(xvb_extractor_t* h, float* const* tables, int ntables, int64_t row0, int64_t ld) {
  XVB_CHECK_ARG(h && h->finalized && ntables >= 0 && ntables <= XVB_MAX_PEERS, "xvb_extractor_set_gather: bad arguments");
  XVB_CHECK_ARG(ntables == 0 || (tables && row0 >= 0 && ld >= h->segment.back().Cout && ld % 4 == 0),
                "xvb_extractor_set_gather: need tables, row0 >= 0, ld >= embed_dim and ld %% 4 == 0");
  for (int k = 0; k < ntables; ++k) h->gather_tables[k] = tables[k];
  h->gather_n = ntables; h->gather_row0 = row0; h->gather_ld = ld;
  return XVB_OK;
}

static bool lanes_enabled() {
  static const int knob = getenv("XVB_LANES") ? atoi(getenv("XVB_LANES")) : 1;
  return knob != 0;
}

// Second lane + the two lane streams, created on first use.
static int ensure_lanes(xvb_extractor* h) {
  if (h->lane1) return XVB_OK;
  for (int i = 0; i < 2; ++i) {
    XVB_CUDA(cudaStreamCreateWithFlags(&h->lane_stream[i], cudaStreamNonBlocking));
    XVB_CUDA(cudaEventCreateWithFlags(&h->ev_lane_done[i], cudaEventDisableTiming));
  }
  XVB_CUDA(cudaEventCreateWithFlags(&h->ev_lane_start, cudaEventDisableTiming));
  xvb_extractor* c = new xvb_extractor();
  c->feat_dim = h->feat_dim; c->ldf = h->ldf; c->finalized = true; c->pooling_eps = h->pooling_eps;
  c->frame = h->frame; c->segment = h->segment;          // Layer = device pointers + shape: shared, not owned
  c->max_c = h->max_c; c->max_seg_c = h->max_seg_c; c->fused_pooling = h->fused_pooling;
  c->im2col_first = h->im2col_first; c->pad_front = h->pad_front; c->pad_back = h->pad_back;
  c->is_lane = true;
  h->lane1 = c;
  return XVB_OK;
}

// fork: both lane streams start after everything already queued on `s`; join: `s` continues after both lanes
static int lanes_fork(xvb_extractor* h, cudaStream_t s) {
  XVB_CUDA(cudaEventRecord(h->ev_lane_start, s));
  for (int i = 0; i < 2; ++i) XVB_CUDA(cudaStreamWaitEvent(h->lane_stream[i], h->ev_lane_start, 0));
  return XVB_OK;
}
static int lanes_join(xvb_extractor* h, cudaStream_t s) {
  for (int i = 0; i < 2; ++i) {
    XVB_CUDA(cudaEventRecord(h->ev_lane_done[i], h->lane_stream[i]));
    XVB_CUDA(cudaStreamWaitEvent(s, h->ev_lane_done[i], 0));
  }
  return XVB_OK;
}

// The caller loop of the reference (extract_embeddings.py:73-83: one utterance per iteration) for a whole
// shard of N equal-length utterances resident on the device: ceil(N / batch) batches through the stack,
// embeddings written in place.  Asynchronous on `stream` (the two lanes fork from it and join it again; with
// per-kernel profiling on, or XVB_LANES=0, the batches run back to back on `stream` itself).
extern "C" int xvb_extractor_extract_shard(xvb_extractor_t* h, const float* feats, int64_t N, int T, int batch, float* emb,
                                           void* stream) {
  XVB_CHECK_ARG(h && h->finalized && feats && emb && N > 0 && T > 0 && batch > 0, "xvb_extractor_extract_shard: bad arguments");
  const int D = h->segment.back().Cout;
  int launches = 0;
  if (lanes_enabled() && !h->profiling && N > batch) {
    int rc = ensure_lanes(h);
    if (rc) return rc;
    if ((rc = lanes_fork(h, (cudaStream_t)stream))) return rc;
    int k = 0;
    for (int64_t i = 0; i < N; i += batch, ++k) {
      const int b = (int)(N - i < batch ? N - i : batch);
      xvb_extractor* lane = (k & 1) ? h->lane1 : h;
      rc = xvb_extractor_extract(lane, feats + (size_t)i * T * h->feat_dim, b, T, emb + (size_t)i * D, h->lane_stream[k & 1]);
      if (rc) return rc;
      launches += lane->last_launches;
      if (h->gather_n) {
        if ((rc = xvb_scatter_rows(emb + (size_t)i * D, b, D, h->gather_tables, h->gather_n, h->gather_row0 + i, h->gather_ld,
                                   h->lane_stream[k & 1]))) return rc;
        ++launches;
      }
    }
    if ((rc = lanes_join(h, (cudaStream_t)stream))) return rc;
    h->last_launches = launches;
    return XVB_OK;
  }
  h->events_used = 0;
  h->in_shard = true;
  for (int64_t i = 0; i < N; i += batch) {
    const int b = (int)(N - i < batch ? N - i : batch);
    int rc = xvb_extractor_extract(h, feats + (size_t)i * T * h->feat_dim, b, T, emb + (size_t)i * D, stream);
    if (!rc && h->gather_n && !h->profiling)
      rc = xvb_scatter_rows(emb + (size_t)i * D, b, D, h->gather_tables, h->gather_n, h->gather_row0 + i, h->gather_ld, stream);
    if (rc) { h->in_shard = false; return rc; }
    launches += h->last_launches;
  }
  h->in_shard = false;
  h->last_launches = launches;
  return XVB_OK;
}

extern "C" int xvb_extractor_extract_host(xvb_extractor_t* h, const float* feats_host, int B, int T, float* emb_host,
                                          void* stream) {
  XVB_CHECK_ARG(h && h->finalized && feats_host && emb_host && B > 0 && T > 0, "xvb_extractor_extract_host: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  const size_t nf = (size_t)B * T * h->feat_dim, ne = (size_t)B * h->segment.back().Cout;
  if (nf > h->h_feats_cap) {
    cudaFree(h->h_feats);
    int rc = dev_alloc(&h->h_feats, nf);
    if (rc) return rc;
    h->h_feats_cap = nf;
  }
  if (ne > h->h_emb_cap) {
    cudaFree(h->h_emb);
    int rc = dev_alloc(&h->h_emb, ne);
    if (rc) return rc;
    h->h_emb_cap = ne;
  }
  XVB_CUDA(cudaMemcpyAsync(h->h_feats, feats_host, nf * sizeof(float), cudaMemcpyHostToDevice, s));
  int rc = xvb_extractor_extract(h, h->h_feats, B, T, h->h_emb, stream);
  if (rc) return rc;
  XVB_CUDA(cudaMemcpyAsync(emb_host, h->h_emb, ne * sizeof(float), cudaMemcpyDeviceToHost, s));
  XVB_CUDA(cudaStreamSynchronize(s));
  return XVB_OK;
}

static int ensure_pipeline(xvb_extractor* h) {
  if (h->copy_stream) return XVB_OK;
  XVB_CUDA(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
  for (int i = 0; i < xvb_extractor::kSlots; ++i) {
    XVB_CUDA(cudaEventCreateWithFlags(&h->ev_h2d[i], cudaEventDisableTiming));
    XVB_CUDA(cudaEventCreateWithFlags(&h->ev_done[i], cudaEventDisableTiming));
  }
  return XVB_OK;
}

static int reserve_slot(xvb_extractor* h, int slot, size_t nf, size_t ne) {
  if (nf > h->p_feats_cap[slot]) {
    cudaFree(h->p_feats[slot]);
    h->p_feats[slot] = nullptr; h->p_feats_cap[slot] = 0;
    int rc = dev_alloc(&h->p_feats[slot], nf);
    if (rc) return rc;
    h->p_feats_cap[slot] = nf;
  }
  if (ne > h->p_emb_cap[slot]) {
    cudaFree(h->p_emb[slot]);
    h->p_emb[slot] = nullptr; h->p_emb_cap[slot] = 0;
    int rc = dev_alloc(&h->p_emb[slot], ne);
    if (rc) return rc;
    h->p_emb_cap[slot] = ne;
  }
  return XVB_OK;
}

extern "C" int xvb_extractor_submit_host(xvb_extractor_t* h, const float* feats_host, int B, int T, float* emb_host,
                                         int slot, void* stream) {
  XVB_CHECK_ARG(h && h->finalized && feats_host && emb_host && B > 0 && T > 0 && (slot == 0 || slot == 1),
                "xvb_extractor_submit_host: bad arguments (slot must be 0 or 1)");
  XVB_CHECK_ARG(!h->slot_busy[slot], "xvb_extractor_submit_host: slot %d still in flight (call xvb_extractor_wait)", slot);
  cudaStream_t s = (cudaStream_t)stream;
  int rc0 = ensure_pipeline(h);
  if (rc0) return rc0;
  const size_t nf = (size_t)B * T * h->feat_dim, ne = (size_t)B * h->segment.back().Cout;
  if ((rc0 = reserve_slot(h, slot, nf, ne))) return rc0;
  // the copy engine fills this slot while the compute stream still works on the other one
  XVB_CUDA(cudaMemcpyAsync(h->p_feats[slot], feats_host, nf * sizeof(float), cudaMemcpyHostToDevice, h->copy_stream));
  XVB_CUDA(cudaEventRecord(h->ev_h2d[slot], h->copy_stream));
  XVB_CUDA(cudaStreamWaitEvent(s, h->ev_h2d[slot], 0));
  int rc = xvb_extractor_extract(h, h->p_feats[slot], B, T, h->p_emb[slot], stream);
  if (rc) return rc;
  XVB_CUDA(cudaMemcpyAsync(emb_host, h->p_emb[slot], ne * sizeof(float), cudaMemcpyDeviceToHost, s));
  XVB_CUDA(cudaEventRecord(h->ev_done[slot], s));
  h->slot_busy[slot] = true;
  return XVB_OK;
}

extern "C" int xvb_extractor_wait(xvb_extractor_t* h, int slot) {
  XVB_CHECK_ARG(h && (slot == 0 || slot == 1), "xvb_extractor_wait: bad arguments");
  if (!h->slot_busy[slot]) return XVB_OK;
  XVB_CUDA(cudaEventSynchronize(h->ev_done[slot]));
  h->slot_busy[slot] = false;
  return XVB_OK;
}

// The same loop end to end through HOST buffers (pinned, so that the copies are asynchronous): batch k's features
// cross the link on the copy stream into one of two device slots while batch k-1 runs; embeddings go back batch by
// batch on `stream`.  No host synchronisation inside the loop (slot reuse is ordered by events on the device);
// returns when the whole shard's embeddings are in `emb_host`.
extern "C" int xvb_extractor_extract_shard_host(xvb_extractor_t* h, const float* feats_host, int64_t N, int T, int batch,
                                                float* emb_host, void* stream) {
  XVB_CHECK_ARG(h && h->finalized && feats_host && emb_host && N > 0 && T > 0 && batch > 0,
                "xvb_extractor_extract_shard_host: bad arguments");
  XVB_CHECK_ARG(!h->slot_busy[0] && !h->slot_busy[1], "xvb_extractor_extract_shard_host: a submit_host slot is still in flight");
  cudaStream_t s = (cudaStream_t)stream;
  int rc;
  if ((rc = ensure_pipeline(h))) return rc;
  const int D = h->segment.back().Cout;
  const int bmax = (int)(N < batch ? N : batch);
  constexpr int S = xvb_extractor::kSlots;
  for (int slot = 0; slot < S; ++slot)
    if ((rc = reserve_slot(h, slot, (size_t)bmax * T * h->feat_dim, (size_t)bmax * D))) return rc;
  // batch k: lane k & 1, device slot k % 4 (two per lane: the copy engine runs up to two batches ahead of a lane); the
  // stack and the copy of the embeddings back run on that lane's stream
  const bool lanes = lanes_enabled() && !h->profiling && N > batch;
  if (lanes) {
    if ((rc = ensure_lanes(h))) return rc;
    if ((rc = lanes_fork(h, s))) return rc;
  }
  int launches = 0, k = 0;
  for (int64_t i = 0; i < N; i += batch, ++k) {
    const int b = (int)(N - i < batch ? N - i : batch);
    const int slot = k % S;
    xvb_extractor* lane = (lanes && (k & 1)) ? h->lane1 : h;
    cudaStream_t ls = lanes ? h->lane_stream[k & 1] : s;
    if (k >= S) XVB_CUDA(cudaStreamWaitEvent(h->copy_stream, h->ev_done[slot], 0));   // batch k-4 has left this slot
    XVB_CUDA(cudaMemcpyAsync(h->p_feats[slot], feats_host + (size_t)i * T * h->feat_dim, (size_t)b * T * h->feat_dim * sizeof(float),
                             cudaMemcpyHostToDevice, h->copy_stream));
    XVB_CUDA(cudaEventRecord(h->ev_h2d[slot], h->copy_stream));
    XVB_CUDA(cudaStreamWaitEvent(ls, h->ev_h2d[slot], 0));
    if ((rc = xvb_extractor_extract(lane, h->p_feats[slot], b, T, h->p_emb[slot], ls))) return rc;
    if (h->gather_n && (rc = xvb_scatter_rows(h->p_emb[slot], b, D, h->gather_tables, h->gather_n, h->gather_row0 + i, h->gather_ld, ls)))
      return rc;
    XVB_CUDA(cudaMemcpyAsync(emb_host + (size_t)i * D, h->p_emb[slot], (size_t)b * D * sizeof(float), cudaMemcpyDeviceToHost, ls));
    XVB_CUDA(cudaEventRecord(h->ev_done[slot], ls));
    launches += lane->last_launches;
  }
  if (lanes && (rc = lanes_join(h, s))) return rc;
  XVB_CUDA(cudaStreamSynchronize(s));
  h->last_launches = launches;
  return XVB_OK;
}

// A shard of N utterances of any lengths through host buffers: xvb_ragged_plan's batches (length-sorted) through the same
// two-lane / four-slot pipeline as xvb_extractor_extract_shard_host.  A batch's utterances are gathered into its device
// slot with one copy per run of consecutive input utterances; its [offsets | lengths] block, uploaded for all batches at
// the start, is copied into the lane's workspace on the lane's stream.  Embeddings come back in batch order and are put
// into input order on the host after the final synchronisation.
extern "C" int xvb_extractor_extract_ragged_shard_host(xvb_extractor_t* h, const float* feats_host, const int64_t* offsets_host,
                                                       int64_t N, int batch, int64_t max_frames, float* emb_host, void* stream) {
  XVB_CHECK_ARG(h && h->finalized && feats_host && offsets_host && emb_host && N > 0 && batch > 0,
                "xvb_extractor_extract_ragged_shard_host: bad arguments");
  XVB_CHECK_ARG(!h->slot_busy[0] && !h->slot_busy[1], "xvb_extractor_extract_ragged_shard_host: a submit_host slot is still in flight");
  int rc = ragged_state_ok(h, "xvb_extractor_extract_ragged_shard_host");
  if (rc) return rc;
  std::vector<int32_t> order((size_t)N);
  std::vector<int64_t> first((size_t)N + 1);
  int64_t nbatch = 0;
  if ((rc = xvb_ragged_plan(offsets_host, N, batch, max_frames, order.data(), first.data(), &nbatch))) return rc;
  const int F = h->feat_dim, D = h->segment.back().Cout;
  // every batch's [offsets (b+1) | lengths (b)] block, offsets relative to the batch's packed features
  std::vector<int32_t> meta;
  meta.reserve((size_t)(2 * N + nbatch));
  std::vector<size_t> meta_at((size_t)nbatch);
  int64_t max_rows = 0, bmax = 0;
  for (int64_t k = 0; k < nbatch; ++k) {
    const int64_t i0 = first[k], i1 = first[k + 1];
    meta_at[k] = meta.size();
    int64_t rows = 0;
    meta.push_back(0);
    for (int64_t i = i0; i < i1; ++i) {
      rows += offsets_host[order[i] + 1] - offsets_host[order[i]];
      XVB_CHECK_ARG(rows <= INT32_MAX, "xvb_extractor_extract_ragged_shard_host: a batch exceeds 2^31 frames");
      meta.push_back((int32_t)rows);
    }
    for (int64_t i = i0; i < i1; ++i) meta.push_back((int32_t)(offsets_host[order[i] + 1] - offsets_host[order[i]]));
    max_rows = std::max(max_rows, rows);
    bmax = std::max(bmax, i1 - i0);
  }
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = ensure_pipeline(h))) return rc;
  constexpr int S = xvb_extractor::kSlots;
  for (int slot = 0; slot < S; ++slot)
    if ((rc = reserve_slot(h, slot, (size_t)max_rows * F, (size_t)bmax * D))) return rc;
  if (meta.size() > h->shard_meta_cap) {
    cudaFree(h->shard_meta);
    h->shard_meta = nullptr; h->shard_meta_cap = 0;
    if ((rc = dev_alloc(&h->shard_meta, meta.size()))) return rc;
    h->shard_meta_cap = meta.size();
  }
  const size_t ne = (size_t)N * D;
  if (ne > h->ragged_emb_host_cap) {
    cudaFreeHost(h->ragged_emb_host);
    h->ragged_emb_host = nullptr; h->ragged_emb_host_cap = 0;
    XVB_CUDA(cudaMallocHost((void**)&h->ragged_emb_host, ne * sizeof(float)));
    h->ragged_emb_host_cap = ne;
  }
  // `meta` outlives the copy: this call returns only after synchronising `stream`
  XVB_CUDA(cudaMemcpyAsync(h->shard_meta, meta.data(), meta.size() * sizeof(int32_t), cudaMemcpyHostToDevice, s));
  const bool lanes = lanes_enabled() && !h->profiling && nbatch > 1;
  if (lanes) {
    if ((rc = ensure_lanes(h))) return rc;
    if ((rc = lanes_fork(h, s))) return rc;
  }
  int launches = 0;
  for (int64_t k = 0; k < nbatch; ++k) {
    const int64_t i0 = first[k];
    const int b = (int)(first[k + 1] - i0);
    const int max_len = meta[meta_at[k] + b + 1 + b - 1];   // the batch is sorted by length: the last one is the longest
    const int Tq = (int)round_up(max_len, kRaggedQuantum);
    const int slot = (int)(k % S);
    xvb_extractor* lane = (lanes && (k & 1)) ? h->lane1 : h;
    cudaStream_t ls = lanes ? h->lane_stream[k & 1] : s;
    if (k >= S) XVB_CUDA(cudaStreamWaitEvent(h->copy_stream, h->ev_done[slot], 0));   // batch k-4 has left this slot
    float* dst = h->p_feats[slot];
    for (int64_t i = i0; i < i0 + b;) {   // runs of consecutive input utterances are contiguous in feats_host
      int64_t j = i + 1;
      while (j < i0 + b && order[j] == order[j - 1] + 1) ++j;
      const int64_t r0 = offsets_host[order[i]], r1 = offsets_host[order[j - 1] + 1];
      XVB_CUDA(cudaMemcpyAsync(dst, feats_host + (size_t)r0 * F, (size_t)(r1 - r0) * F * sizeof(float), cudaMemcpyHostToDevice,
                               h->copy_stream));
      dst += (size_t)(r1 - r0) * F;
      i = j;
    }
    XVB_CUDA(cudaEventRecord(h->ev_h2d[slot], h->copy_stream));
    XVB_CUDA(cudaStreamWaitEvent(ls, h->ev_h2d[slot], 0));
    if ((rc = reserve(lane, b, Tq))) return rc;
    XVB_CUDA(cudaMemcpyAsync(lane->ragged_meta, h->shard_meta + meta_at[k], (size_t)(2 * b + 1) * sizeof(int32_t),
                             cudaMemcpyDeviceToDevice, ls));
    if ((rc = run_stack(lane, h->p_feats[slot], b, Tq, true, h->p_emb[slot], ls))) return rc;
    XVB_CUDA(cudaMemcpyAsync(h->ragged_emb_host + (size_t)i0 * D, h->p_emb[slot], (size_t)b * D * sizeof(float),
                             cudaMemcpyDeviceToHost, ls));
    XVB_CUDA(cudaEventRecord(h->ev_done[slot], ls));
    launches += lane->last_launches;
  }
  if (lanes && (rc = lanes_join(h, s))) return rc;
  XVB_CUDA(cudaStreamSynchronize(s));
  for (int64_t i = 0; i < N; ++i)
    memcpy(emb_host + (size_t)order[i] * D, h->ragged_emb_host + (size_t)i * D, (size_t)D * sizeof(float));
  h->last_launches = launches;
  return XVB_OK;
}

extern "C" int xvb_extractor_set_fused_pooling(xvb_extractor_t* h, int enable) {
  XVB_CHECK_ARG(h, "xvb_extractor_set_fused_pooling: null extractor");
  if (h->fused_pooling != (enable != 0)) h->drop_plans();
  h->fused_pooling = enable != 0;
  if (h->lane1) return xvb_extractor_set_fused_pooling(h->lane1, enable);
  return XVB_OK;
}

extern "C" int xvb_extractor_set_profiling(xvb_extractor_t* h, int enable) {
  XVB_CHECK_ARG(h, "xvb_extractor_set_profiling: null extractor");
  h->profiling = enable != 0;
  h->events_used = 0;
  return XVB_OK;
}

extern "C" int xvb_extractor_kernel_times(xvb_extractor_t* h, float* ms_host, int max_n) {
  XVB_CHECK_ARG(h && ms_host, "xvb_extractor_kernel_times: null argument");
  if (h->events_used < 2) return 0;
  XVB_CUDA(cudaEventSynchronize(h->events[h->events_used - 1]));
  int n = h->events_used - 1;
  if (n > max_n) n = max_n;
  for (int i = 0; i < n; ++i) XVB_CUDA(cudaEventElapsedTime(&ms_host[i], h->events[i], h->events[i + 1]));
  return n;
}

extern "C" int xvb_extractor_last_launches(const xvb_extractor_t* h) { return h ? h->last_launches : XVB_ESTATE; }

extern "C" const float* xvb_extractor_debug_f32(const xvb_extractor_t* h, int which) {
  if (!h) return nullptr;
  return which < 0 ? h->stats : h->last_f32;
}

extern "C" void xvb_extractor_destroy(xvb_extractor_t* h) {
  if (!h) return;
  if (h->lane1) xvb_extractor_destroy(h->lane1);
  for (int i = 0; i < 2; ++i) {
    if (h->lane_stream[i]) cudaStreamDestroy(h->lane_stream[i]);
    if (h->ev_lane_done[i]) cudaEventDestroy(h->ev_lane_done[i]);
  }
  if (h->ev_lane_start) cudaEventDestroy(h->ev_lane_start);
  h->free_ws();
  for (cudaEvent_t e : h->events) cudaEventDestroy(e);
  for (int i = 0; i < xvb_extractor::kSlots; ++i) {
    cudaFree(h->p_feats[i]); cudaFree(h->p_emb[i]);
    if (h->ev_h2d[i]) cudaEventDestroy(h->ev_h2d[i]);
    if (h->ev_done[i]) cudaEventDestroy(h->ev_done[i]);
  }
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  if (h->ev_meta) cudaEventDestroy(h->ev_meta);
  cudaFreeHost(h->ragged_meta_host); cudaFreeHost(h->ragged_emb_host); cudaFree(h->shard_meta);
  cudaFree(h->h_feats); cudaFree(h->h_emb); cudaFree(h->pool_partial);
  if (!h->is_lane)
    for (auto* v : {&h->frame, &h->segment})
      for (Layer& L : *v) { cudaFree(L.w_hi); cudaFree(L.w_lo); cudaFree(L.bias); cudaFree(L.scale); cudaFree(L.shift); }
  delete h;
}
