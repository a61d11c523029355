// C ABI of libavh_b200.so (include/avh_b200.h): handle, weight folding/repacking, per-shape execution plans
// and the forward orchestration of AVHubertModel.extract_finetune (avhubert/hubert.py:694-745) on sm_100a.
//
// Data layout in HBM (N = B*T tokens/frames, P = 1 in bf16 mode, 2 (hi|mid bf16 planes) in fp32 mode):
//   lip frontend activations   NHWC with one shared zero row/column per image: [n, H+1, W+1, C]; a 3x3/s1
//                              conv is then 9 row-shifted GEMM taps over the flat [n*(H+1)*(W+1), C] matrix
//                              (TMA out-of-bounds zero fill covers the first/last image)
//   tokens                     row-major [N, C]; residual stream in fp32, GEMM operands bf16 [N, P*C]
//   positional-conv input      [B*(T+64), P*D] bf16 with 64 zero rows after every clip (time halo)
//   weights                    K-major bf16 [out, P*K] (conv: K = (kh,kw,cin); pos-conv: K = (tap, window))
#include "avh_b200.h"
#include "common.cuh"
#include "gemm.h"
#include "kernels.h"

#include <array>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <tuple>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include <cuda_fp16.h>

namespace avh {

static thread_local std::string g_err;
void set_last_error(const std::string& msg) { g_err = msg; }
static std::atomic<long long> g_launches{0};
static std::atomic<long long> g_graph_launches{0};      // cudaGraphLaunch calls (avh_graph_launch_count)
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

bool pdl_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = std::getenv("AVH_PDL");
    v = (e != nullptr && e[0] == '0') ? 0 : 1;
  }
  return v != 0;
}

int device_sm_count() {
  static int cached_dev = -1, cached_n = 148;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev != cached_dev) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) cached_n = n;
    cached_dev = dev;
  }
  return cached_n;
}

int ensure_dyn_smem(const void* fn, int bytes) {
  static std::mutex mu;
  static std::map<std::pair<int, const void*>, int> done;      // (device, function) -> bytes granted
  int dev = 0;
  AVH_CUDA_OK(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(mu);
  auto it = done.find({dev, fn});
  if (it != done.end() && it->second >= bytes) return 0;
  AVH_CUDA_OK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  done[{dev, fn}] = bytes;
  return 0;
}

namespace {

typedef __nv_bfloat16 bf16;

struct HostTensor {
  std::vector<float> v;
  std::vector<int64_t> shape;
  int64_t numel() const { return (int64_t)v.size(); }
};

// ---------------------------------------------------------------------------- device memory arena
struct Arena {
  char* base = nullptr;
  size_t cap = 0, used = 0;
  int init(size_t bytes) {
    cap = bytes;
    AVH_CUDA_OK(cudaMalloc(&base, cap));
    AVH_CUDA_OK(cudaMemset(base, 0, cap));
    return 0;
  }
  void* take(size_t bytes) {
    used = (used + 1023) & ~(size_t)1023;
    void* p = base + used;
    used += bytes;
    return used <= cap ? p : nullptr;
  }
  void release() {
    if (base) cudaFree(base);
    base = nullptr;
  }
};
// two-pass allocation: first pass sizes the arena (base == nullptr), second pass hands out pointers
struct Sizer {
  size_t used = 0;
  void take(size_t bytes) {
    used = (used + 1023) & ~(size_t)1023;
    used += bytes;
  }
};

inline bf16 f2bf(float x) { return __float2bfloat16_rn(x); }
inline float bf2f(bf16 x) { return __bfloat162float(x); }

// ---------------------------------------------------------------------------- packed weights
struct PackedW {          // K-major bf16 [n, P*kpad] on the device
  bf16* w = nullptr;
  int n = 0, k = 0, kpad = 0;
};
struct ConvUnit {         // conv + folded eval-mode BatchNorm (+ PReLU)
  PackedW w;
  float* scale = nullptr;
  float* bias = nullptr;
  float* slope = nullptr;
  // training-mode BatchNorm: affine parameters and the running statistics the batch statistics update (device, fp32)
  float *gamma = nullptr, *beta = nullptr, *rmean = nullptr, *rvar = nullptr;
  int cin = 0, cout = 0, ks = 3, stride = 1;
  PackedW wT;               // trainable handles: [K = ks*ks*cin rows, cout] — the B operand of d_col = d_raw W
};
struct BlockW {
  ConvUnit c1, c2, ds;
  bool has_ds = false;
  float* slope2 = nullptr;
  // bf16 frame-row path: conv2 and the 1x1 shortcut conv in ONE GEMM — weights [cout, 9*cout + cin] with both
  // BatchNorm scales folded in, bias = b2 + b_ds, scale = 1
  PackedW c2ds;
  float* c2ds_bias = nullptr;
  float* ones = nullptr;
};
struct LinearW {
  PackedW w;
  float* bias = nullptr;
};
struct LayerW {
  LinearW qkv, out, fc1, fc2;
  // W^T packed K-major (rows = in features, K = out features): the B operand of dX = dY W in the backward pass; only
  // packed for trainable handles (cfg.reserved[3] != 0), bias pointers unused
  LinearW qkvT, outT, fc1T, fc2T;
  float *ln1_g = nullptr, *ln1_b = nullptr, *ln2_g = nullptr, *ln2_b = nullptr;
};

// Q-Former (src/sub_model/Qformer.py) handle: BERT-style post-LN layers over the query tokens, each = self-attention,
// cross-attention to the AV features, feed-forward with the *_query weights
struct QfLayerW {
  LinearW sqkv, sout, cq, cout, fc1, fc2;
  float *ln1_g = nullptr, *ln1_b = nullptr, *ln2_g = nullptr, *ln2_b = nullptr, *ln3_g = nullptr, *ln3_b = nullptr;
};

struct Step {
  std::function<int(cudaStream_t)> run;
  std::string name;       // kernel class for avh_profile_json
  double flops = 0;       // executed tensor-core FLOPs (GEMM steps)
  int layer = -1;         // encoder layer the step belongs to (LayerDrop skips it in training mode), -1 = none
  bool direct = false;    // reads or writes a CALLER pointer (video, audio, features, output): never part of a CUDA graph
  bool on_drop = false;   // runs only when its layer is dropped (the identity that stands in for the layer)
  int mod = 0;            // modality dropout: 1 audio / 2 video arm of the step (skipped when that modality is dropped;
                          // an on_drop step runs only then), 0 = none
};

struct CallArgs {          // per-call pointers the steps read through the plan
  const void* video = nullptr;
  int video_dt = 0;
  const void* audio = nullptr;
  int audio_dt = 0;
  long long as[3] = {0, 0, 0};
  const unsigned char* mask = nullptr;
  void* out = nullptr;
  int out_dt = 0;
  const void* xin = nullptr; // encoder-only plans: features [B,T,D]
  int xin_dt = 0;
  int pitch = 0;             // ragged plans: time pitch of the caller's padded tensors (baked into captured launches)
  void* grads_out = nullptr; // training backward: the caller's gradient buffer, filled bucket by bucket (never captured)
  int grads_dt = 0;
};

enum class PlanKind {
  Forward,        // avh_forward: AVHubertModel.extract_finetune
  // avh_forward_ragged: packed ragged batches.  Every buffer holds Nb = round_up(sum of clip lengths, 128) token /
  // frame rows with the clips back to back; T is then the longest clip the plan serves (attention tiling).  The
  // per-call geometry lives in a small device descriptor `rag` (int32): [0] stem work items, [1] rows in use,
  // [16..16+B] first row of every clip (cu), then the stem's (clip, band, t0, t1) item list.
  Ragged,
  EncoderOnly,    // avh_encoder_forward: TransformerEncoder on caller-provided features [B,T,D]
  // avh_forward_train: BatchNorm batch statistics through the generic convolution path, Philox dropout at the
  // reference's dropout sites, LayerDrop by skipping a layer's launches; never graph-captured
  TrainForward,
  // training plans (forward with saved activations + backward, avh_encoder_backward): steps [0, fwd_steps) are the
  // forward, the rest the backward; gradients accumulate in a plan-owned fp32 buffer
  EncoderTrain,   // TransformerEncoder on caller-provided features
  TailTrain,      // trainable tail of AV-HuBERT (fusion LayerNorm + post_extract_proj + encoder) on caller-provided fused features
  FullTrain,      // the whole model (lip ResNet + projections computed in the plan, feature_grad_mult > 0)
  QFormer,        // avh_qformer_forward: T = query rows per clip, Lk = AV feature rows per clip
};

// One plan (= workspace + launch list) per key: shape, inputs present, kind AND CUDA stream.  Forwards enqueued on
// different streams never share scratch memory, so a caller can keep several batches in flight on one device.
struct PlanKey {
  PlanKind kind = PlanKind::Forward;
  int B = 0, T = 0;
  bool has_video = false, has_audio = false, has_mask = false;
  int output_layer = 0;
  long long ragged_rows = 0;      // Ragged: Nb
  int Lk = 0;                     // QFormer
  cudaStream_t stream = nullptr;
  // training plans (avh_set_train_args): dropout_input (tail modes), dropout, activation_dropout, and whether the
  // caller draws LayerDrop coins; all 0 / false: the launch list of a step without regularisation
  float p_in = 0.f, p_enc = 0.f, p_act = 0.f;
  bool layerdrop = false;
  // pretraining steps (avh_set_modality_drop): the plan can drop a modality (TrainForward / FullTrain with both
  // modalities), and the FullTrain backward adds the features_pen gradient to dL/d(fused); both false: the launch list
  // of a fine-tuning step
  bool moddrop = false, pen = false;
  bool training() const { return kind == PlanKind::EncoderTrain || kind == PlanKind::TailTrain || kind == PlanKind::FullTrain; }
  bool dropout() const { return p_in > 0.f || p_enc > 0.f || p_act > 0.f; }
  bool operator<(const PlanKey& o) const {
    return std::tie(kind, B, T, has_video, has_audio, has_mask, output_layer, ragged_rows, Lk, stream, p_in, p_enc, p_act,
                    layerdrop, moddrop, pen) <
           std::tie(o.kind, o.B, o.T, o.has_video, o.has_audio, o.has_mask, o.output_layer, o.ragged_rows, o.Lk, o.stream, o.p_in,
                    o.p_enc, o.p_act, o.layerdrop, o.moddrop, o.pen);
  }
};

struct Plan {
  PlanKey key;
  float p_in = 0.f, p_enc = 0.f, p_act = 0.f, bn_momentum = 0.1f;     // training-mode forward: set per call
  unsigned long long seed = 0;
  std::vector<unsigned char> layer_skip;
  int mod_drop = 0;                // modality dropped by the current step (key.moddrop plans): 0 none, 1 audio, 2 video
  float* dpen = nullptr;           // key.pen plans: dL/dfeatures_pen of the current step (device word, avh_set_features_pen_grad)
  const void* fused_buf = nullptr; // fused features [B*T, E] of the last forward (avh_train_features_pen)
  int fused_dt = 0;
  size_t fwd_steps = 0;
  float* grads = nullptr;
  long long grad_floats = 0;
  float* dx_out = nullptr;         // gradient w.r.t. the input features [B*T, D] fp32
  float* dy_in = nullptr;          // gradient w.r.t. the output, staged fp32 [B*T, D]
  float fgm = 1.f;                 // mode 2: feature_grad_mult (GradMultiply on the extractor outputs), set per call
  bool fwd_done = false;
  unsigned char* qmask_dev = nullptr;    // Q-Former plans: [B*T] 1 = padded query, [B*Lk] 1 = padded AV frame
  unsigned char* kmask_dev = nullptr;
  int* rag = nullptr;
  int rag_ints = 0, rag_items_off = 0, rag_max_items = 0;
  static constexpr int RAG_SLOTS = 4;
  int* rag_host[RAG_SLOTS] = {nullptr, nullptr, nullptr, nullptr};      // pinned mirrors, used round robin
  cudaEvent_t rag_done[RAG_SLOTS] = {nullptr, nullptr, nullptr, nullptr};
  // training plans: gradient buckets in the order the backward completes them ([begin, end) floats of the flat buffer)
  // and one event per bucket, recorded right after the bucket was copied into the caller's buffer
  struct GradBucket { long long begin, end; cudaEvent_t ev; };
  std::vector<GradBucket> buckets;
  int rag_next = 0;
  // training plans with dropout: the seed of the current step in a device word the kernels read (captured graphs
  // replay for any seed), written from pinned mirrors used round robin like rag_host
  unsigned long long* seed_dev = nullptr;
  unsigned long long* seed_host[RAG_SLOTS] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t seed_done[RAG_SLOTS] = {nullptr, nullptr, nullptr, nullptr};
  int seed_next = 0;
  int* pos_row_map = nullptr;

  Arena arena;
  std::vector<Step> steps;
  std::vector<GemmPlan*> gemms;
  std::vector<ConvWinPlan*> convwins;
  std::vector<ConvFramePlan*> convframes;
  StemFusedPlan stemf;
  AttnTcPlan att;
  std::map<std::string, std::pair<const void*, std::pair<int, long long>>> stages;   // name -> (ptr, (dtype, numel))
  CallArgs args;
  // CUDA graphs of the launch list (all steps but the last, which writes the caller's output and is launched
  // directly), one per distinct set of INPUT pointers (kernel arguments are baked in at capture).  A forward is ~200
  // launches = ~3 ms of host time — as long as the GPU needs for the step; a graph launch is one driver call.
  // Framework allocators hand the same addresses back for same-shaped tensors and the host-buffer entry point always
  // runs from its own staging buffers, so the cache hits after the first calls; a caller that never repeats an
  // address stops being captured (captures/calls guard) and gets plain launches.
  // Segmented graphs: every maximal run of steps that touch only plan-owned memory is one CUDA graph, captured on the
  // second forward and replayed ever after whatever tensors the caller passes — the few steps that read the caller's
  // video / audio / feature pointers or write its output are launched directly in between, and the padding mask is
  // copied into a plan-owned buffer first (B*T bytes).  (Round 1 keyed whole-forward graphs on the input pointers: a
  // caller with fresh tensors per batch never hit the cache and paid ~3 ms of host enqueue per 3.9 ms step.)
  struct Segment { size_t begin, end; cudaGraphExec_t exec; int kernels; };
  std::vector<Segment> segments;
  bool segments_ready = false;
  unsigned char* mask_dev = nullptr;   // staged copy of the caller's padding mask [B*T]
  int direct_runs = 0;              // un-captured forwards so far (the first one also configures the kernels)
  long long last_use = 0;           // LRU clock value of the most recent forward through this plan
  void drop_graphs() {
    for (auto& sg : segments)
      if (sg.exec) cudaGraphExecDestroy(sg.exec);
    segments.clear();
    segments_ready = false;
  }
  ~Plan() {
    drop_graphs();
    for (GemmPlan* g : gemms) delete g;
    for (ConvWinPlan* g : convwins) delete g;
    for (ConvFramePlan* g : convframes) delete g;
    for (int i = 0; i < RAG_SLOTS; ++i) {
      if (rag_host[i]) cudaFreeHost(rag_host[i]);
      if (rag_done[i]) cudaEventDestroy(rag_done[i]);
      if (seed_host[i]) cudaFreeHost(seed_host[i]);
      if (seed_done[i]) cudaEventDestroy(seed_done[i]);
    }
    for (GradBucket& gb : buckets)
      if (gb.ev) cudaEventDestroy(gb.ev);
    arena.release();
  }
};

}  // namespace
}  // namespace avh

using namespace avh;

struct avh_handle {
  avh_config cfg;
  int device = 0;
  int P = 1;                       // operand planes: 1 = bf16, 2 = fp32-faithful split
  bool finalized = false;
  std::map<std::string, HostTensor> raw;
  Arena warena;
  ConvUnit stem;
  PackedW stem_wf;          // stem weights in the K order of the fused kernel (stem_fused.cu)
  BlockW blocks[4][2];
  LinearW proj_v, proj_a, post_proj;
  LinearW post_projT;             // trainable handles: post_extract_proj^T for the backward
  LinearW proj_vT;                // ... and feature_extractor_video.proj^T (gradient into the ResNet features)
  bool has_post_proj = false;
  float *fuse_ln_g = nullptr, *fuse_ln_b = nullptr, *enc_ln_g = nullptr, *enc_ln_b = nullptr;
  PackedW pos_w;
  PackedW pos_wT;                 // trainable handles: the same windowed layout with in / out swapped inside every group
  float *pos_v_raw = nullptr, *pos_g_raw = nullptr;     // trainable handles: weight_v [D, D/G, KT], weight_g [KT] (fp32)
  float* pos_bias = nullptr;
  int pos_window = 64;            // input-channel window per 64-column N tile (64 or 128)
  int* pos_acol = nullptr;        // device [D/64] window start per N tile
  float* pos_ratio = nullptr;     // trainable handles: device scratch [KT] of the weight-norm ratios (refresh on the device)
  // trainable handles: how every packed tensor the TRAINING plans read derives from a state-dict entry, recorded by the
  // packers; avh_refresh_weights_device replays the list with device kernels (refresh.cu)
  struct RefreshJob {
    std::string src;              // state-dict key
    int form = 0;                 // RJ_*
    void* dst = nullptr;
    long long n = 0, k = 0;       // source [n, k] (matrix forms), n elements (vector), cout / cin (conv)
    long long ld = 0;             // elements of one plane of a destination row
    long long off = 0;            // destination row offset (matrix), column offset (transposed matrix)
    float scale = 1.f;
    int ks = 0;                   // conv: taps per side
  };
  std::vector<RefreshJob> refresh_jobs;
  // the job list captured as one CUDA graph for the parameter pointers it was last called with (an optimizer updates the
  // same tensors in place every step: ~650 small launches become one graph launch)
  std::vector<long long> refresh_key;
  cudaGraphExec_t refresh_exec = nullptr;
  // every AV-HuBERT handle: how the EVAL-only packed forms derive from BatchNorm parameters and buffers and conv
  // weights, recorded by the packers; avh_refresh_eval_weights_device replays the list (after the training-form jobs)
  // with device kernels, captured as its own graph for the pointer set it was last called with
  struct EvalJob {
    std::string bn;               // fold: BatchNorm prefix of ".weight", ".bias", ".running_mean", ".running_var"
    ConvUnit* cu = nullptr;       // fold: writes cu->scale, bias, gamma, beta, rmean, rvar
    BlockW* bw = nullptr;         // c2ds: writes bw->c2ds and c2ds_bias from the folds of bw->c2 and bw->ds (earlier jobs)
    std::string w2, wd;           // c2ds: state-dict keys of conv2 and downsample.0 weights
  };
  std::vector<EvalJob> eval_jobs;
  std::vector<long long> eval_refresh_key;
  cudaGraphExec_t eval_refresh_exec = nullptr;
  std::vector<LayerW> layers;
  // Q-Former handles (cfg.reserved[0] == 2): reserved[1] = encoder_width, reserved[2] = rows of query_tokens
  std::vector<QfLayerW> qf_layers;
  LinearW qf_ckv;                  // cross-attention key / value projections of ALL layers: [L * 2D, encoder_width]
  float *qf_emb_g = nullptr, *qf_emb_b = nullptr, *qf_tokens = nullptr;
  std::map<PlanKey, std::unique_ptr<Plan>> plans;
  long long plan_clock = 0;
  bool profiling = false;
  std::vector<cudaEvent_t> prof_events;      // 2 per step of the last profiled forward
  Plan* prof_plan = nullptr;
  Plan* last_plan = nullptr;      // plan of the most recent avh_forward (avh_read_stage reads its stages)
  struct Staging {                // device staging of avh_forward_host, one set per stream
    void* video = nullptr; void* audio = nullptr; void* mask = nullptr; void* out = nullptr;
    void* video_pp = nullptr;     // normalised + cropped frames when the caller hands raw uint8 video
    size_t video_cap = 0, audio_cap = 0, mask_cap = 0, out_cap = 0, video_pp_cap = 0;
  };
  std::map<void*, Staging> staging;
  // raw-video geometry and normalisation for video_dtype == AVH_U8 (avh_set_video_preprocess)
  int vp_src_h = 88, vp_src_w = 88;
  double vp_mean = 0.421, vp_std = 0.165;
  // avh_set_train_args: regularisation of the next training step on this handle, consumed by it
  struct NextTrain {
    float p_in = 0.f, p_enc = 0.f, p_act = 0.f;
    unsigned long long seed = 0;
    std::vector<unsigned char> skip;      // LayerDrop coins (1 = dropped); empty = LayerDrop off
  };
  NextTrain next_train;
  // avh_set_modality_drop: the next training forward is a pretraining step dropping this modality (0 none, 1 audio,
  // 2 video); -1 = not a pretraining step
  int next_mod_drop = -1;
};

namespace avh {
namespace {

int dtype_size(int dt) { return dt == AVH_F32 ? 4 : (dt == AVH_U8 ? 1 : 2); }

// ============================================================================ weight folding / packing
enum { RJ_MATRIX = 0, RJ_MATRIX_T, RJ_VEC, RJ_CONV, RJ_CONV_T, RJ_STEM, RJ_POS, RJ_POS_T, RJ_VEC_OFF };

struct Packer {
  avh_handle* h;
  Arena* arena;      // null during sizing
  Sizer sizer;
  std::string missing;

  const HostTensor* get(const std::string& key) {
    auto it = h->raw.find(key);
    if (it == h->raw.end()) {
      if (missing.empty()) missing = key;
      return nullptr;
    }
    return &it->second;
  }
  template <typename T>
  T* upload(const std::vector<T>& host) {
    const size_t bytes = host.size() * sizeof(T);
    if (arena == nullptr) {
      sizer.take(bytes);
      return nullptr;
    }
    T* d = reinterpret_cast<T*>(arena->take(bytes));
    if (d == nullptr) return nullptr;
    if (cudaMemcpy(d, host.data(), bytes, cudaMemcpyHostToDevice) != cudaSuccess) return nullptr;
    return d;
  }
  // fp32 [n, kpad] -> bf16 planes [n, P*kpad]
  PackedW pack(const std::vector<float>& w, int n, int k, int kpad) {
    const int P = h->P;
    PackedW out;
    out.n = n; out.k = k; out.kpad = kpad;
    if (arena == nullptr) {
      sizer.take((size_t)n * P * kpad * sizeof(bf16));
      return out;
    }
    std::vector<bf16> host((size_t)n * P * kpad);
    for (int r = 0; r < n; ++r)
      for (int c = 0; c < kpad; ++c) {
        const float x = w[(size_t)r * kpad + c];
        const bf16 hi = f2bf(x);
        host[(size_t)r * P * kpad + c] = hi;
        if (P > 1) host[(size_t)r * P * kpad + kpad + c] = f2bf(x - bf2f(hi));
      }
    out.w = upload(host);
    return out;
  }
  float* upload_f(const std::vector<float>& v) { return upload(v); }
  // record how a packed destination derives from a state-dict entry (trainable handles, real pass only)
  bool recording() const { return arena != nullptr && h->cfg.reserved[3] != 0; }
  void job(const std::string& src, int form, void* dst, long long n, long long k, long long ld, long long off = 0, float scale = 1.f,
           int ks = 0) {
    if (!recording() || dst == nullptr) return;
    avh_handle::RefreshJob j;
    j.src = src; j.form = form; j.dst = dst; j.n = n; j.k = k; j.ld = ld; j.off = off; j.scale = scale; j.ks = ks;
    h->refresh_jobs.push_back(j);
  }
  void job_vec(const std::string& src, float* dst, long long n, float scale = 1.f) { job(src, RJ_VEC, dst, n, 0, 0, 0, scale); }
  // eval-only forms (every handle, real pass only)
  void eval_fold(const std::string& bn, ConvUnit* cu) {
    if (arena == nullptr) return;
    avh_handle::EvalJob j;
    j.bn = bn; j.cu = cu;
    h->eval_jobs.push_back(j);
  }
  void eval_c2ds(const std::string& w2, const std::string& wd, BlockW* bw) {
    if (arena == nullptr) return;
    avh_handle::EvalJob j;
    j.bw = bw; j.w2 = w2; j.wd = wd;
    h->eval_jobs.push_back(j);
  }
};

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// conv weight [cout, cin, kh, kw] (+ BN) -> K-major [(kh,kw,cin)] + folded scale/bias
bool pack_conv(Packer& pk, const std::string& wkey, const std::string& bnkey, const std::string& prelu_key,
               int ks, int stride, ConvUnit* cu) {
  const HostTensor* w = pk.get(wkey);
  const HostTensor* g = pk.get(bnkey + ".weight");
  const HostTensor* b = pk.get(bnkey + ".bias");
  const HostTensor* m = pk.get(bnkey + ".running_mean");
  const HostTensor* v = pk.get(bnkey + ".running_var");
  const HostTensor* s = prelu_key.empty() ? nullptr : pk.get(prelu_key);
  if (!w || !g || !b || !m || !v || (!prelu_key.empty() && !s)) return false;
  const int cout = (int)w->shape[0], cin = (int)w->shape[1];
  cu->cin = cin; cu->cout = cout; cu->ks = ks; cu->stride = stride;
  const int K = ks * ks * cin;
  std::vector<float> packed((size_t)cout * K);
  for (int o = 0; o < cout; ++o)
    for (int c = 0; c < cin; ++c)
      for (int t = 0; t < ks * ks; ++t) packed[(size_t)o * K + (size_t)t * cin + c] = w->v[((size_t)o * cin + c) * ks * ks + t];
  cu->w = pk.pack(packed, cout, K, K);
  pk.job(wkey, RJ_CONV, cu->w.w, cout, cin, K, 0, 1.f, ks);
  if (pk.h->cfg.reserved[3] != 0 && pk.h->cfg.reserved[0] == 0) {
    const int cp = round_up(cout, 64);
    std::vector<float> pt((size_t)K * cp, 0.f);
    for (int o = 0; o < cout; ++o)
      for (int k = 0; k < K; ++k) pt[(size_t)k * cp + o] = packed[(size_t)o * K + k];
    cu->wT = pk.pack(pt, K, cout, cp);
    pk.job(wkey, RJ_CONV_T, cu->wT.w, cout, cin, cp, 0, 1.f, ks);
  }
  std::vector<float> sc(cout), bi(cout);
  for (int o = 0; o < cout; ++o) {
    const float inv = 1.0f / std::sqrt(v->v[o] + 1e-5f);      // nn.BatchNorm eps default
    sc[o] = g->v[o] * inv;
    bi[o] = b->v[o] - m->v[o] * sc[o];
  }
  cu->scale = pk.upload_f(sc);
  cu->bias = pk.upload_f(bi);
  cu->gamma = pk.upload_f(g->v); cu->beta = pk.upload_f(b->v);
  cu->rmean = pk.upload_f(m->v); cu->rvar = pk.upload_f(v->v);
  pk.eval_fold(bnkey, cu);
  pk.job_vec(bnkey + ".weight", cu->gamma, cout);
  pk.job_vec(bnkey + ".bias", cu->beta, cout);
  cu->slope = nullptr;
  if (s) {
    std::vector<float> sl(cout);
    for (int o = 0; o < cout; ++o) sl[o] = s->v[s->numel() == 1 ? 0 : o];
    cu->slope = pk.upload_f(sl);
    pk.job_vec(prelu_key, cu->slope, cout);
  }
  return true;
}

// the transpose of a packed Linear: [k, n] with K = n (zero padded to 64)
bool pack_linear_T(Packer& pk, const std::vector<std::string>& prefixes, const std::vector<float>& scales, LinearW* lw) {
  int k = -1, n = 0;
  std::vector<const HostTensor*> ws;
  for (const std::string& pre : prefixes) {
    const HostTensor* w = pk.get(pre + ".weight");
    if (!w) return false;
    if (k < 0) k = (int)w->shape[1];
    n += (int)w->shape[0];
    ws.push_back(w);
  }
  const int npad = (n + 63) / 64 * 64;
  std::vector<float> p((size_t)k * npad, 0.f);
  int r0 = 0;
  for (size_t t = 0; t < ws.size(); ++t) {
    const int nn = (int)ws[t]->shape[0];
    for (int r = 0; r < nn; ++r)
      for (int c = 0; c < k; ++c) p[(size_t)c * npad + r0 + r] = ws[t]->v[(size_t)r * k + c] * scales[t];
    r0 += nn;
  }
  lw->w = pk.pack(p, k, n, npad);
  lw->bias = nullptr;
  r0 = 0;
  for (size_t t = 0; t < ws.size(); ++t) {
    pk.job(prefixes[t] + ".weight", RJ_MATRIX_T, lw->w.w, ws[t]->shape[0], k, npad, r0, scales[t]);
    r0 += (int)ws[t]->shape[0];
  }
  return true;
}

bool pack_linear(Packer& pk, const std::string& prefix, LinearW* lw, float wscale = 1.f) {
  const HostTensor* w = pk.get(prefix + ".weight");
  const HostTensor* b = pk.get(prefix + ".bias");
  if (!w || !b) return false;
  const int n = (int)w->shape[0], k = (int)w->shape[1], kpad = round_up(k, 64);
  std::vector<float> p((size_t)n * kpad, 0.f);
  for (int r = 0; r < n; ++r)
    for (int c = 0; c < k; ++c) p[(size_t)r * kpad + c] = w->v[(size_t)r * k + c] * wscale;
  lw->w = pk.pack(p, n, k, kpad);
  std::vector<float> bb(b->v);
  for (auto& x : bb) x *= wscale;
  lw->bias = pk.upload_f(bb);
  pk.job(prefix + ".weight", RJ_MATRIX, lw->w.w, n, k, kpad, 0, wscale);
  pk.job_vec(prefix + ".bias", lw->bias, n, wscale);
  return true;
}

// several nn.Linear with the same input stacked along the output dim (fused q / k / v, the K / V of all layers)
bool pack_linear_cat(Packer& pk, const std::vector<std::string>& prefixes, LinearW* lw) {
  std::vector<float> wcat, bcat;
  int k = -1, n = 0;
  for (const std::string& pre : prefixes) {
    const HostTensor* w = pk.get(pre + ".weight");
    const HostTensor* b = pk.get(pre + ".bias");
    if (!w || !b) return false;
    if (k < 0) k = (int)w->shape[1];
    if ((int)w->shape[1] != k) return false;
    wcat.insert(wcat.end(), w->v.begin(), w->v.end());
    bcat.insert(bcat.end(), b->v.begin(), b->v.end());
    n += (int)w->shape[0];
  }
  const int kpad = round_up(k, 64);
  std::vector<float> p((size_t)n * kpad, 0.f);
  for (int r = 0; r < n; ++r)
    for (int c = 0; c < k; ++c) p[(size_t)r * kpad + c] = wcat[(size_t)r * k + c];
  lw->w = pk.pack(p, n, k, kpad);
  lw->bias = pk.upload_f(bcat);
  return true;
}

// Q-Former weights, BertModel-level key names (src/sub_model/Qformer.py:52-111,379-486) + "query_tokens"
bool pack_qformer(Packer& pk) {
  avh_handle* h = pk.h;
  const int L = h->cfg.encoder_layers;
  bool ok = true;
  auto ln = [&](const std::string& pre, float** g, float** b) {
    const HostTensor* gw = pk.get(pre + ".weight");
    const HostTensor* bw = pk.get(pre + ".bias");
    if (gw && bw) { *g = pk.upload_f(gw->v); *b = pk.upload_f(bw->v); } else ok = false;
  };
  ln("embeddings.LayerNorm", &h->qf_emb_g, &h->qf_emb_b);
  const HostTensor* qt = pk.get("query_tokens");
  if (qt) h->qf_tokens = pk.upload_f(qt->v); else ok = false;
  h->qf_layers.resize(L);
  std::vector<std::string> kv;
  for (int l = 0; l < L; ++l) {
    const std::string pre = "encoder.layer." + std::to_string(l) + ".";
    QfLayerW& lw = h->qf_layers[l];
    ok &= pack_linear_cat(pk, {pre + "attention.self.query", pre + "attention.self.key", pre + "attention.self.value"}, &lw.sqkv);
    ok &= pack_linear(pk, pre + "attention.output.dense", &lw.sout);
    ln(pre + "attention.output.LayerNorm", &lw.ln1_g, &lw.ln1_b);
    ok &= pack_linear(pk, pre + "crossattention.self.query", &lw.cq);
    kv.push_back(pre + "crossattention.self.key");
    kv.push_back(pre + "crossattention.self.value");
    ok &= pack_linear(pk, pre + "crossattention.output.dense", &lw.cout);
    ln(pre + "crossattention.output.LayerNorm", &lw.ln2_g, &lw.ln2_b);
    ok &= pack_linear(pk, pre + "intermediate_query.dense", &lw.fc1);
    ok &= pack_linear(pk, pre + "output_query.dense", &lw.fc2);
    ln(pre + "output_query.LayerNorm", &lw.ln3_g, &lw.ln3_b);
  }
  ok &= pack_linear_cat(pk, kv, &h->qf_ckv);
  return ok;
}

bool pack_all(Packer& pk) {
  avh_handle* h = pk.h;
  const avh_config& c = h->cfg;
  if (c.reserved[0] == 2) return pack_qformer(pk);
  const int D = c.encoder_embed_dim;
  const std::string R = "feature_extractor_video.resnet.";
  bool ok = true;
  const bool enc_only = c.reserved[0] != 0;      // handle of a bare TransformerEncoder (avh_encoder_forward only)
  // ---- stem: Conv3d weight [64,1,5,7,7] -> [64, 5*64]
  if (!enc_only) {
    const HostTensor* w = pk.get(R + "frontend3D.0.weight");
    const HostTensor* g = pk.get(R + "frontend3D.1.weight");
    const HostTensor* b = pk.get(R + "frontend3D.1.bias");
    const HostTensor* m = pk.get(R + "frontend3D.1.running_mean");
    const HostTensor* v = pk.get(R + "frontend3D.1.running_var");
    const HostTensor* s = pk.get(R + "frontend3D.2.weight");
    if (w && g && b && m && v && s) {
      std::vector<float> p((size_t)64 * 320, 0.f);      // K = dt*64 + kh*7 + kw (49..63 of each tap zero)
      for (int o = 0; o < 64; ++o)
        for (int dt = 0; dt < 5; ++dt)
          for (int k = 0; k < 49; ++k) p[(size_t)o * 320 + dt * 64 + k] = w->v[(size_t)o * 245 + dt * 49 + k];
      h->stem.w = pk.pack(p, 64, 245, 320);
      pk.job(R + "frontend3D.0.weight", RJ_STEM, h->stem.w.w, 64, 245, 320);
      std::vector<float> pf((size_t)64 * 320, 0.f);     // fused stem kernel: K = dt*64 + kh*8 + kw
      for (int o = 0; o < 64; ++o)
        for (int dt = 0; dt < 5; ++dt)
          for (int kh = 0; kh < 7; ++kh)
            for (int kw = 0; kw < 7; ++kw)
              pf[(size_t)o * 320 + dt * 64 + kh * 8 + kw] = w->v[(size_t)o * 245 + dt * 49 + kh * 7 + kw];
      h->stem_wf = pk.pack(pf, 64, 320, 320);
      pk.job(R + "frontend3D.0.weight", RJ_STEM, h->stem_wf.w, 64, 245, 320, 0, 1.f, 8);      // ks = 8: the kh*8 + kw order
      h->stem.cin = 1; h->stem.cout = 64;
      std::vector<float> sc(64), bi(64), sl(64);
      for (int o = 0; o < 64; ++o) {
        const float inv = 1.0f / std::sqrt(v->v[o] + 1e-5f);
        sc[o] = g->v[o] * inv;
        bi[o] = b->v[o] - m->v[o] * sc[o];
        sl[o] = s->v[s->numel() == 1 ? 0 : o];
      }
      h->stem.scale = pk.upload_f(sc);
      h->stem.bias = pk.upload_f(bi);
      h->stem.slope = pk.upload_f(sl);
      h->stem.gamma = pk.upload_f(g->v); h->stem.beta = pk.upload_f(b->v);
      h->stem.rmean = pk.upload_f(m->v); h->stem.rvar = pk.upload_f(v->v);
      pk.eval_fold(R + "frontend3D.1", &h->stem);
      pk.job_vec(R + "frontend3D.1.weight", h->stem.gamma, 64);
      pk.job_vec(R + "frontend3D.1.bias", h->stem.beta, 64);
      pk.job_vec(R + "frontend3D.2.weight", h->stem.slope, 64);
    } else ok = false;
  }
  // ---- ResNet-18 trunk (avhubert/resnet.py:77-129)
  for (int L = 0; L < (enc_only ? 0 : 4); ++L)
    for (int bi = 0; bi < 2; ++bi) {
      BlockW& bw = h->blocks[L][bi];
      const std::string pre = R + "trunk.layer" + std::to_string(L + 1) + "." + std::to_string(bi) + ".";
      const int stride = (L > 0 && bi == 0) ? 2 : 1;
      ok &= pack_conv(pk, pre + "conv1.weight", pre + "bn1", pre + "relu1.weight", 3, stride, &bw.c1);
      ok &= pack_conv(pk, pre + "conv2.weight", pre + "bn2", "", 3, 1, &bw.c2);
      bw.has_ds = (L > 0 && bi == 0);
      if (bw.has_ds) ok &= pack_conv(pk, pre + "downsample.0.weight", pre + "downsample.1", "", 1, stride, &bw.ds);
      if (bw.has_ds) {
        const HostTensor* w2 = pk.get(pre + "conv2.weight");
        const HostTensor* wd = pk.get(pre + "downsample.0.weight");
        auto bn_fold = [&](const std::string& bn, std::vector<float>* sc, std::vector<float>* bi) {
          const HostTensor* g = pk.get(bn + ".weight");
          const HostTensor* b = pk.get(bn + ".bias");
          const HostTensor* m = pk.get(bn + ".running_mean");
          const HostTensor* v = pk.get(bn + ".running_var");
          if (!g || !b || !m || !v) return false;
          sc->resize(g->v.size()); bi->resize(g->v.size());
          for (size_t o = 0; o < g->v.size(); ++o) {
            const float inv = 1.0f / std::sqrt(v->v[o] + 1e-5f);
            (*sc)[o] = g->v[o] * inv;
            (*bi)[o] = b->v[o] - m->v[o] * (*sc)[o];
          }
          return true;
        };
        std::vector<float> s2v, b2v, sdv, bdv;
        if (w2 && wd && bn_fold(pre + "bn2", &s2v, &b2v) && bn_fold(pre + "downsample.1", &sdv, &bdv)) {
          const int cout = (int)w2->shape[0], cmid = (int)w2->shape[1], cin = (int)wd->shape[1];
          const int K = 9 * cmid + cin;
          std::vector<float> packed((size_t)cout * K), bias(cout), ones(cout, 1.0f);
          for (int o = 0; o < cout; ++o) {
            for (int c = 0; c < cmid; ++c)
              for (int t = 0; t < 9; ++t)
                packed[(size_t)o * K + (size_t)t * cmid + c] = s2v[o] * w2->v[((size_t)o * cmid + c) * 9 + t];
            for (int c = 0; c < cin; ++c) packed[(size_t)o * K + 9 * cmid + c] = sdv[o] * wd->v[(size_t)o * cin + c];
            bias[o] = b2v[o] + bdv[o];
          }
          bw.c2ds = pk.pack(packed, cout, K, K);
          bw.c2ds_bias = pk.upload_f(bias);
          bw.ones = pk.upload_f(ones);
          pk.eval_c2ds(pre + "conv2.weight", pre + "downsample.0.weight", &bw);
        } else ok = false;
      }
      const HostTensor* s2 = pk.get(pre + "relu2.weight");
      if (s2) {
        const int cout = 64 << L;
        std::vector<float> sl(cout);
        for (int o = 0; o < cout; ++o) sl[o] = s2->v[s2->numel() == 1 ? 0 : o];
        bw.slope2 = pk.upload_f(sl);
        pk.job_vec(pre + "relu2.weight", bw.slope2, cout);
      } else ok = false;
    }
  // ---- modality projections, fusion LN, post_extract_proj
  if (!enc_only) {
    ok &= pack_linear(pk, "feature_extractor_video.proj", &h->proj_v);
    if (c.reserved[3] != 0) ok &= pack_linear_T(pk, {"feature_extractor_video.proj"}, {1.f}, &h->proj_vT);
    ok &= pack_linear(pk, "feature_extractor_audio.proj", &h->proj_a);
    const HostTensor* g = pk.get("layer_norm.weight");
    const HostTensor* b = pk.get("layer_norm.bias");
    if (g && b) {
      h->fuse_ln_g = pk.upload_f(g->v); h->fuse_ln_b = pk.upload_f(b->v);
      pk.job_vec("layer_norm.weight", h->fuse_ln_g, (long long)g->v.size());
      pk.job_vec("layer_norm.bias", h->fuse_ln_b, (long long)b->v.size());
    } else ok = false;
  }
  h->has_post_proj = !enc_only && (c.modality_fuse == AVH_FUSE_CONCAT);
  if (h->has_post_proj) ok &= pack_linear(pk, "post_extract_proj", &h->post_proj);
  if (h->has_post_proj && c.reserved[3] != 0) ok &= pack_linear_T(pk, {"post_extract_proj"}, {1.f}, &h->post_projT);
  // ---- positional conv: weight-norm(dim=2) fold, grouped -> per-N-tile windowed dense K-major
  {
    const HostTensor* wg = pk.get("encoder.pos_conv.0.weight_g");
    const HostTensor* wv = pk.get("encoder.pos_conv.0.weight_v");
    const HostTensor* wb = pk.get("encoder.pos_conv.0.bias");
    if (wg && wv && wb) {
      const int KT = c.conv_pos, G = c.conv_pos_groups, cg = D / G;    // taps, groups, channels per group
      // norm over (out, in) per tap (torch.nn.utils.weight_norm dim=2, wav2vec2.py:834)
      std::vector<double> nrm(KT, 0.0);
      for (size_t i = 0; i < wv->v.size(); ++i) nrm[i % KT] += (double)wv->v[i] * wv->v[i];
      std::vector<float> ratio(KT);
      for (int k = 0; k < KT; ++k) ratio[k] = (float)((double)wg->v[k] / std::sqrt(nrm[k]));
      const int ntile = D / 64;
      std::vector<int> acol(ntile);
      int window = 64;
      for (int j = 0; j < ntile; ++j) {
        const int g0 = (64 * j) / cg, g1 = (64 * j + 63) / cg;
        acol[j] = g0 * cg;
        const int need = (g1 + 1) * cg - g0 * cg;
        if (need > window) window = round_up(need, 64);
      }
      h->pos_window = window;
      const int kpad = KT * window;
      std::vector<float> p((size_t)D * kpad, 0.f);
      for (int o = 0; o < D; ++o) {
        const int g = o / cg, j = o / 64;
        for (int i = 0; i < cg; ++i) {
          const int col = g * cg + i - acol[j];           // position inside the tile's window
          for (int k = 0; k < KT; ++k)
            p[(size_t)o * kpad + (size_t)k * window + col] = wv->v[((size_t)o * cg + i) * KT + k] * ratio[k];
        }
      }
      h->pos_w = pk.pack(p, D, kpad, kpad);
      h->pos_bias = pk.upload_f(wb->v);
      h->pos_acol = pk.upload(acol);
      pk.job("encoder.pos_conv.0.weight_v", RJ_POS, h->pos_w.w, D, cg, kpad);
      pk.job_vec("encoder.pos_conv.0.bias", h->pos_bias, D);
      if (c.reserved[3] != 0) {
        // backward w.r.t. the input: dx[t, i] = sum_k sum_o dc[t + KT/2 - k, o] w[o, i, k] — row = input channel, the
        // window holds the OUTPUT channels of the same groups (groups cover the same channel range on both sides)
        std::vector<float> pt((size_t)D * kpad, 0.f);
        for (int o = 0; o < D; ++o) {
          const int g = o / cg;
          for (int i = 0; i < cg; ++i) {
            const int ig = g * cg + i, j = ig / 64;
            const int col = o - acol[j];
            for (int k = 0; k < KT; ++k)
              pt[(size_t)ig * kpad + (size_t)k * window + col] = wv->v[((size_t)o * cg + i) * KT + k] * ratio[k];
          }
        }
        h->pos_wT = pk.pack(pt, D, kpad, kpad);
        h->pos_v_raw = pk.upload_f(wv->v);
        h->pos_g_raw = pk.upload_f(wg->v);
        h->pos_ratio = pk.upload_f(ratio);
        pk.job("encoder.pos_conv.0.weight_v", RJ_POS_T, h->pos_wT.w, D, cg, kpad);
        pk.job_vec("encoder.pos_conv.0.weight_v", h->pos_v_raw, (long long)wv->v.size());
        pk.job_vec("encoder.pos_conv.0.weight_g", h->pos_g_raw, (long long)wg->v.size());
      }
    } else ok = false;
  }
  // ---- transformer layers: fused QKV with q scaling folded (multihead_attention.py:60, scaling = hd^-0.5)
  h->layers.resize(c.encoder_layers);
  const float qscale = 1.0f / std::sqrt((float)(D / c.encoder_attention_heads));
  for (int l = 0; l < c.encoder_layers; ++l) {
    LayerW& lw = h->layers[l];
    const std::string pre = "encoder.layers." + std::to_string(l) + ".";
    const HostTensor* qw = pk.get(pre + "self_attn.q_proj.weight");
    const HostTensor* kw = pk.get(pre + "self_attn.k_proj.weight");
    const HostTensor* vw = pk.get(pre + "self_attn.v_proj.weight");
    const HostTensor* qb = pk.get(pre + "self_attn.q_proj.bias");
    const HostTensor* kb = pk.get(pre + "self_attn.k_proj.bias");
    const HostTensor* vb = pk.get(pre + "self_attn.v_proj.bias");
    if (qw && kw && vw && qb && kb && vb) {
      std::vector<float> w((size_t)3 * D * D), b((size_t)3 * D);
      for (size_t i = 0; i < (size_t)D * D; ++i) {
        w[i] = qw->v[i] * qscale;
        w[(size_t)D * D + i] = kw->v[i];
        w[(size_t)2 * D * D + i] = vw->v[i];
      }
      for (int i = 0; i < D; ++i) { b[i] = qb->v[i] * qscale; b[D + i] = kb->v[i]; b[2 * D + i] = vb->v[i]; }
      lw.qkv.w = pk.pack(w, 3 * D, D, D);
      lw.qkv.bias = pk.upload_f(b);
      {
        const char* nm[3] = {"self_attn.q_proj", "self_attn.k_proj", "self_attn.v_proj"};
        for (int t = 0; t < 3; ++t) {
          pk.job(pre + nm[t] + ".weight", RJ_MATRIX, lw.qkv.w.w, D, D, D, (long long)t * D, t == 0 ? qscale : 1.f);
          pk.job(pre + nm[t] + ".bias", RJ_VEC_OFF, lw.qkv.bias, D, 0, 0, (long long)t * D, t == 0 ? qscale : 1.f);
        }
      }
    } else ok = false;
    ok &= pack_linear(pk, pre + "self_attn.out_proj", &lw.out);
    ok &= pack_linear(pk, pre + "fc1", &lw.fc1);
    ok &= pack_linear(pk, pre + "fc2", &lw.fc2);
    if (c.reserved[3] != 0) {      // trainable handle: W^T operands of the dgrad GEMMs (avh_encoder_backward)
      ok &= pack_linear_T(pk, {pre + "self_attn.q_proj", pre + "self_attn.k_proj", pre + "self_attn.v_proj"},
                          {qscale, 1.f, 1.f}, &lw.qkvT);
      ok &= pack_linear_T(pk, {pre + "self_attn.out_proj"}, {1.f}, &lw.outT);
      ok &= pack_linear_T(pk, {pre + "fc1"}, {1.f}, &lw.fc1T);
      ok &= pack_linear_T(pk, {pre + "fc2"}, {1.f}, &lw.fc2T);
    }
    const HostTensor* g1 = pk.get(pre + "self_attn_layer_norm.weight");
    const HostTensor* b1 = pk.get(pre + "self_attn_layer_norm.bias");
    const HostTensor* g2 = pk.get(pre + "final_layer_norm.weight");
    const HostTensor* b2 = pk.get(pre + "final_layer_norm.bias");
    if (g1 && b1 && g2 && b2) {
      lw.ln1_g = pk.upload_f(g1->v); lw.ln1_b = pk.upload_f(b1->v);
      lw.ln2_g = pk.upload_f(g2->v); lw.ln2_b = pk.upload_f(b2->v);
      pk.job_vec(pre + "self_attn_layer_norm.weight", lw.ln1_g, D);
      pk.job_vec(pre + "self_attn_layer_norm.bias", lw.ln1_b, D);
      pk.job_vec(pre + "final_layer_norm.weight", lw.ln2_g, D);
      pk.job_vec(pre + "final_layer_norm.bias", lw.ln2_b, D);
    } else ok = false;
  }
  {
    const HostTensor* g = pk.get("encoder.layer_norm.weight");
    const HostTensor* b = pk.get("encoder.layer_norm.bias");
    if (g && b) {
      h->enc_ln_g = pk.upload_f(g->v); h->enc_ln_b = pk.upload_f(b->v);
      pk.job_vec("encoder.layer_norm.weight", h->enc_ln_g, D);
      pk.job_vec("encoder.layer_norm.bias", h->enc_ln_b, D);
    } else ok = false;
  }
  return ok;
}

// ============================================================================ plan construction
struct Tap {
  int a_row_off, a_col, b_col;
};

// GEMM epilogue writing [M, N] rows of stride ldc (fp32 or bf16); the other fields are filled per call site
Epilogue epilogue(void* C, long long ldc, bool c_fp32) {
  Epilogue ep;
  ep.C = C; ep.ldc = ldc; ep.c_fp32 = c_fp32 ? 1 : 0;
  return ep;
}

// activation tensor: `data` holds the values ([rows, C], bf16 in bf16 mode / fp32 in fp32 mode); `op` is the
// GEMM-operand form (bf16 [rows, P*C]); identical to data in bf16 mode.
struct Act {
  void* data = nullptr;
  void* op = nullptr;
  long long rows = 0;
  int C = 0;
};

struct Builder {
  avh_handle* h;
  Plan* plan;
  bool sizing;
  Sizer sizer;
  int P;
  bool f32;      // fp32-faithful mode
  size_t es;     // bytes per activation value
  int act_dt;    // dtype of activation values
  bool linear_k = false;         // next gemm(): plain K loop without a step table (bf16 mode, single zero tap)
  int force_sk = 0;              // next gemm(): GemmProblem::streamk
  float* sk_ws = nullptr;        // stream-K workspace of the plan's GEMMs (launches of a plan are serialised on its stream)
  size_t sk_bytes = 0;
  int* sk_flags = nullptr;
  int cur_layer = -1;           // encoder layer of the steps pushed next (LayerDrop skips a dropped layer's steps)
  int cur_mod = 0;              // modality arm of the steps pushed next (modality dropout skips a dropped arm's steps)

  Builder(avh_handle* h_, Plan* plan_, bool sizing_)
      : h(h_), plan(plan_), sizing(sizing_), P(h_->P), f32(h_->cfg.compute_mode == AVH_COMPUTE_FP32) {
    es = f32 ? 4 : 2;
    act_dt = f32 ? DT_F32 : DT_BF16;
  }

  void* alloc(size_t bytes) {
    if (sizing) {
      sizer.take(bytes);
      return reinterpret_cast<void*>(0x1000);   // placeholder, never dereferenced
    }
    return plan->arena.take(bytes);
  }
  float* f32buf(long long n) { return reinterpret_cast<float*>(alloc((size_t)n * 4)); }
  Act act(long long rows, int C) {
    Act a;
    a.rows = rows; a.C = C;
    a.data = alloc((size_t)rows * C * es);
    a.op = f32 ? alloc((size_t)rows * C * 2 * P) : a.data;
    return a;
  }
  // plan-owned copy of a [rows] byte mask (padding masks are staged into it before the launch list runs)
  unsigned char* mask_buf(long long rows) { return reinterpret_cast<unsigned char*>(alloc((size_t)rows + 16)); }
  // stream-K workspace: one fp32 partial tile (128 x 256) per SM + flags (zero from the arena's initial fill; the
  // kernels hand the flags back as zeros)
  void stream_k_workspace() {
    sk_bytes = (size_t)device_sm_count() * 128 * 256 * 4;
    sk_ws = f32buf((long long)sk_bytes / 4);
    sk_flags = reinterpret_cast<int*>(alloc(4096));
  }
  void stage(const char* name, const void* p, int dt, long long n) {
    if (!sizing) plan->stages[name] = {p, {dt, n}};
  }

  // `direct`: the step reads or writes caller pointers, so it is launched outside the CUDA graphs
  void push(const std::string& tag, std::function<int(cudaStream_t)> f, double flops = 0.0, bool direct = false) {
    if (!sizing) plan->steps.push_back(Step{std::move(f), tag, flops, cur_layer, direct, false, cur_mod});
  }
  void push_direct(const std::string& tag, std::function<int(cudaStream_t)> f, double flops = 0.0) {
    push(tag, std::move(f), flops, true);
  }
  // a step of layer cur_layer (or of modality arm cur_mod) that runs only when LayerDrop drops that layer (modality
  // dropout that arm), launched directly, between the graphs around it
  void push_on_drop(const std::string& tag, std::function<int(cudaStream_t)> f) {
    if (!sizing) plan->steps.push_back(Step{std::move(f), tag, 0.0, cur_layer, true, true, cur_mod});
  }
  // dropped modality arm: zero `cols` columns of fused rows [rows, ld] (elements of es bytes) from column `off`
  void zero_cols_on_drop(int mod, void* base, long long rows, int ld, int off, int cols, size_t elem) {
    cur_mod = mod;
    char* p = reinterpret_cast<char*>(base) + (size_t)off * elem;
    push_on_drop("modality_drop", [=](cudaStream_t s) {
      return cudaMemset2DAsync(p, (size_t)ld * elem, 0, (size_t)cols * elem, (size_t)rows, s) == cudaSuccess ? 0 : 1;
    });
    cur_mod = 0;
  }
  // fp32 [rows, C] (row stride ld) -> GEMM-operand form (bf16 [rows, P*C])
  void split(const float* src, int ld, void* dst, long long rows, int C) {
    const int planes = P;
    push("split", [=](cudaStream_t s) { return launch_split_rows(src, ld, dst, planes, rows, C, 0, 0, s); });
  }
  // fp32 mode: refresh the split bf16 operand planes of an activation (bf16 mode: op is data)
  void sync_op(const Act& a) {
    if (f32) split(reinterpret_cast<const float*>(a.data), a.C, a.op, a.rows, a.C);
  }
  // LayerNorm over the rows of src ([dst.rows, dst.C] of dtype src_dt) into an activation and its operand form
  void layernorm(const std::string& tag, const void* src, int src_dt, const float* g, const float* be, float eps,
                 const Act& dst) {
    float* of = f32 ? reinterpret_cast<float*>(dst.data) : nullptr;
    void* ol = f32 ? nullptr : dst.data;
    const long long rows = dst.rows;
    const int C = dst.C;
    push(tag, [=](cudaStream_t s) { return launch_layernorm(src, src_dt, C, g, be, eps, of, ol, DT_BF16, nullptr, rows, C, s); });
    sync_op(dst);
  }

  // K-step table for one GEMM: every tap x every 64-wide K chunk (x 3 split-precision products in fp32 mode)
  const KStep* ktable(const std::vector<Tap>& taps, int chunks, int a_plane_stride, int b_plane_stride,
                      int* num_kb) {
    std::vector<KStep> t;
    const int nprod = f32 ? 3 : 1;
    static const int PA[3] = {0, 0, 1}, PB[3] = {0, 1, 0};
    for (int pr = nprod - 1; pr >= 0; --pr)       // small cross terms first, hi*hi last
      for (const Tap& tp : taps)
        for (int c = 0; c < chunks; ++c)
          t.push_back(KStep{tp.a_col + PA[pr] * a_plane_stride + c * 64, tp.a_row_off,
                            tp.b_col + PB[pr] * b_plane_stride + c * 64, 0});
    *num_kb = (int)t.size();
    KStep* d = reinterpret_cast<KStep*>(alloc(t.size() * sizeof(KStep)));
    if (!sizing) cudaMemcpy(d, t.data(), t.size() * sizeof(KStep), cudaMemcpyHostToDevice);
    return d;
  }

  // enqueue one GEMM; returns false on planning failure
  bool gemm(const std::string& tag, const void* A, long long a_rows, int a_cols, const PackedW& W, long long M,
            const std::vector<Tap>& taps, int chunks, int a_plane_stride, const Epilogue& ep, int block_n = 0,
            const int* a_col_nblk = nullptr, long long lda = 0) {
    GemmProblem pr;
    pr.A = A; pr.a_rows = a_rows; pr.a_cols = a_cols; pr.lda = lda > 0 ? lda : a_cols;
    pr.B = W.w; pr.b_rows = W.n; pr.b_cols = P * W.kpad; pr.ldb = (long long)P * W.kpad;
    pr.M = M; pr.N = W.n;
    if (linear_k && !f32 && taps.size() == 1 && taps[0].a_col == 0 && taps[0].a_row_off == 0 && taps[0].b_col == 0) {
      pr.ktable = nullptr;          // K step kb reads columns 64 kb of both operands: no table, no limit on the K extent
      pr.num_kb = chunks;
    } else {
      pr.ktable = ktable(taps, chunks, a_plane_stride, W.kpad, &pr.num_kb);
    }
    pr.streamk = force_sk;
    pr.a_col_nblk = a_col_nblk;
    pr.block_n = block_n;
    pr.sk_ws = sk_ws; pr.sk_ws_bytes = sk_bytes; pr.sk_flags = sk_flags;
    pr.ep = ep;
    if (sizing) return true;
    GemmPlan* gp = new GemmPlan();
    plan->gemms.push_back(gp);
    if (gemm_plan(pr, gp)) return false;
    push(tag, [gp](cudaStream_t s) { return gemm_launch(*gp, s); }, 2.0 * (double)M * (double)W.n * 64.0 * (double)pr.num_kb);
    return true;
  }
  // dense single-tap GEMM: A [rows, P*K] (operand form) x W^T
  bool linear(const std::string& tag, const void* A, long long rows, int K, const PackedW& W, const Epilogue& ep) {
    return gemm(tag, A, rows, P * K, W, rows, {Tap{0, 0, 0}}, K / 64, K, ep);
  }
};

struct FrontendBufs {
  void* im2col = nullptr;   // stem (kh,kw) patches [CB*(T+2)*1936, P*64]
  void* stem_out = nullptr; // [CF*1936, 64]
  Act pooled;               // padded 23x23x64
  Act a[4][4];              // per layer: block0.conv1 out, block0 out, block1.conv1 out, block1 out
  Act ds[4];                // downsample outputs (layers 2-4)
  void* col[4] = {nullptr, nullptr, nullptr, nullptr};   // im2col_s2 outputs (layers 2-4)
};

bool build_plan(avh_handle* h, Plan* plan, bool sizing, size_t* bytes_out) {
  Builder b(h, plan, sizing);
  const avh_config& c = h->cfg;
  const PlanKey& key = plan->key;
  const int P = b.P;
  const bool f32 = b.f32;
  const int B = key.B, T = key.T, D = c.encoder_embed_dim, F = c.encoder_ffn_embed_dim;
  const int Hh = c.encoder_attention_heads;
  const bool rg = key.kind == PlanKind::Ragged;
  const bool enc_only = key.kind == PlanKind::EncoderOnly;
  const bool train = key.kind == PlanKind::TrainForward;
  const bool hm = key.has_mask;
  const long long N = rg ? key.ragged_rows : (long long)B * T;
  const int E = c.modality_fuse == AVH_FUSE_CONCAT ? 2 * D : D;
  const size_t es = b.es;
  const int act_dt = b.act_dt;
  Plan* pl = plan;

  b.stream_k_workspace();
  {
    unsigned char* md = b.mask_buf((long long)B * T);
    if (!sizing) plan->mask_dev = md;
  }
  // fused token features [N, E]: audio arm in columns [0,D), video arm in [D,2D) (concat) or summed (add)
  Act fused = b.act(N, E);
  if (rg) {
    plan->rag_items_off = 16 + ((B + 1 + 3) / 4) * 4;
    plan->rag_max_items = 11 * (int)(N / 2 + B);
    plan->rag_ints = plan->rag_items_off + 4 * plan->rag_max_items;
    int* r = reinterpret_cast<int*>(b.alloc((size_t)plan->rag_ints * 4));
    if (!sizing) plan->rag = r;
  }
  const int v_off = c.modality_fuse == AVH_FUSE_CONCAT ? D : 0;
  const int a_off = 0;

  // ========================================================================== lip frontend
  if (key.has_video) {
    // chunks of whole clips (the stem's temporal taps are row shifts inside a clip-padded layout)
    const int target = c.frontend_chunk_frames > 0 ? c.frontend_chunk_frames : 2400;
    int CB = std::max(1, target / T);
    CB = (B + ((B + CB - 1) / CB) - 1) / ((B + CB - 1) / CB);       // even split over ceil(B/CB) chunks
    if (rg) CB = B;                                                  // ragged: one chunk of Nb packed frames
    // training mode: one chunk, so that BatchNorm normalises with the statistics of the whole batch and updates the
    // running statistics once per forward, as nn.BatchNorm does
    if (train) {
      if ((long long)B * T > 65535) {      // the stem max-pool runs one grid row per frame
        set_last_error("training-mode forward: B*T = " + std::to_string((long long)B * T) +
                       " frames exceed the 65535 frames BatchNorm can take in one frontend pass");
        return false;
      }
      CB = B;
    }
    const int CF = rg ? (int)N : CB * T;
    FrontendBufs fb;
    if (f32 || train) {     // patch matrix + un-pooled stem maps: only the unfused stem needs them
      fb.im2col = b.alloc((size_t)CB * (T + 2) * 1936 * 64 * 2 * P);
      fb.stem_out = b.alloc((size_t)CB * (T + 2) * 1936 * 64 * es);      // same clip-padded row space as the patches
    }
    static const int HS[4] = {22, 11, 6, 3};
    fb.pooled = b.act((long long)CF * 23 * 23, 64);
    for (int L = 0; L < 4; ++L) {
      const int S = HS[L] + 1, Cc = 64 << L;
      for (int i = 0; i < 4; ++i) fb.a[L][i] = b.act((long long)CF * S * S, Cc);
      if (L > 0) {
        fb.ds[L] = b.act((long long)CF * S * S, Cc);
        fb.col[L] = b.alloc((size_t)CF * HS[L] * HS[L] * 9 * (Cc / 2) * P * 2);
      }
    }
    Act pooled_feat = b.act(N, 512);     // avgpool output = ResEncoder output [B*T, 512]
    b.stage("resnet", pooled_feat.data, act_dt, N * 512);

    // ---- training mode: BatchNorm with batch statistics.  The convolution writes its raw output into a scratch map of
    // the output's own layout, bn_stats / bn_finalize produce scale + bias (and update the running statistics),
    // bn_apply does what the eval-mode epilogue fuses (train_ops.cu; avhubert/resnet.py:23,44,56,139)
    void* bn_raw = nullptr;
    double* bn_sums = nullptr;
    float *bn_scale = nullptr, *bn_bias = nullptr;
    if (train) {
      bn_raw = b.alloc((size_t)CB * (T + 2) * 1936 * 64 * es);          // the stem's map is the largest
      bn_sums = reinterpret_cast<double*>(b.alloc((size_t)BN_SLOTS * 2 * 512 * sizeof(double)));
      bn_scale = b.f32buf(512);
      bn_bias = b.f32buf(512);
    }
    // launch(ep) enqueues the convolution with epilogue `ep`; in training mode it is called with a raw epilogue
    auto conv_bn = [&](Epilogue ep, const ConvUnit& cu, long long out_rows, double count, long long period, long long valid,
                       int S, int Himg, const std::function<bool(const Epilogue&)>& launch) -> bool {
      if (!train) return launch(ep);
      Epilogue raw = ep;
      raw.C = bn_raw;
      raw.col_scale = nullptr; raw.col_bias = nullptr; raw.act = ACT_NONE; raw.slope1 = nullptr;
      raw.R = nullptr; raw.slope2 = nullptr;
      if (!launch(raw)) return false;
      const int Cc = cu.cout;
      void* outp = ep.C;
      const float* s1 = ep.act == ACT_PRELU ? ep.slope1 : nullptr;
      const void* res = ep.R;
      const float* s2 = ep.slope2;
      const float *gm = cu.gamma, *bt = cu.beta;
      float *rm = cu.rmean, *rv = cu.rvar;
      b.push("bn_train", [=](cudaStream_t s) {
        return launch_bn_stats(bn_raw, act_dt, out_rows, Cc, period, valid, S, Himg, bn_sums, s);
      });
      b.push("bn_train", [=](cudaStream_t s) {
        return launch_bn_finalize(bn_sums, count, gm, bt, 1e-5f, pl->bn_momentum, rm, rv, bn_scale, bn_bias, Cc, s);
      });
      b.push("bn_train", [=](cudaStream_t s) {
        return launch_bn_apply(bn_raw, outp, act_dt, out_rows, Cc, bn_scale, bn_bias, s1, res, s2, S, Himg, s);
      });
      return true;
    };

    // 3x3 stride-1 conv over the padded layout as 9 shifted taps
    auto conv3x3_s1 = [&](const Act& in, const ConvUnit& cu, const Act& out, int Himg, int nimg, const float* slope1,
                          const Act* res, const float* slope2) -> bool {
      const int S = Himg + 1;
      if (!f32 && !train && cu.cin == 64 && cu.cout == 64) {
        // layer1: operand window resident in smem, nine taps as descriptor row offsets (conv_window.cu)
        if (sizing) return true;
        ConvWinProblem wp;
        wp.A = in.op; wp.B = cu.w.w; wp.rows = (long long)nimg * S * S; wp.S = S;
        wp.scale = cu.scale; wp.bias = cu.bias; wp.slope1 = slope1;
        wp.R = res ? res->data : nullptr; wp.slope2 = slope2; wp.C = out.data;
        ConvWinPlan* cp = new ConvWinPlan();
        plan->convwins.push_back(cp);
        if (conv_window_plan(wp, cp)) return false;
        b.push("conv3x3_c64", [cp](cudaStream_t s) { return conv_window_launch(*cp, s); }, 2.0 * (double)wp.rows * 64.0 * 576.0);
        return true;
      }
      std::vector<Tap> taps;
      for (int kh = 0; kh < 3; ++kh)
        for (int kw = 0; kw < 3; ++kw)
          taps.push_back(Tap{(kh - 1) * S + (kw - 1), 0, (kh * 3 + kw) * cu.cin});
      Epilogue ep = epilogue(out.data, cu.cout, f32);
      ep.col_scale = cu.scale; ep.col_bias = cu.bias;
      if (slope1) { ep.act = ACT_PRELU; ep.slope1 = slope1; }
      if (res) { ep.R = res->data; ep.ldr = cu.cout; ep.r_fp32 = f32 ? 1 : 0; }
      ep.slope2 = slope2;
      ep.map_mode = MAP_2LEVEL; ep.S2 = S * S; ep.S1 = S; ep.H = Himg; ep.W = Himg;
      ep.O2 = S * S; ep.O1 = S; ep.O0 = 0; ep.invalid_zero = 1;
      const long long rows = (long long)nimg * S * S;
      const std::string tag = "conv3x3_c" + std::to_string(cu.cin);
      const void* a_op = in.op;
      const int a_cols = P * cu.cin, chunks = cu.cin / 64, aps = cu.cin;
      if (!conv_bn(ep, cu, rows, (double)nimg * Himg * Himg, 0, 0, S, Himg, [&](const Epilogue& e) {
            return b.gemm(tag, a_op, rows, a_cols, cu.w, rows, taps, chunks, aps, e);
          }))
        return false;
      b.sync_op(out);
      return true;
    };

    // bf16 mode, layers 2-4: one frame per GEMM row, dense [frames, H*H*C] maps, in-image taps only (conv_frame.cu)
    const bool frame_mode = !f32 && !train;
    struct Shortcut { const void* A2 = nullptr; int Cin = 0, Sin = 0, stride = 1; const PackedW* w = nullptr;
                      const float* bias = nullptr; const float* ones = nullptr; };
    auto conv_frame = [&](const void* in, int Hin, int Sin, int Cin, const ConvUnit& cu, void* out, int Hout, int nimg,
                          const float* slope1, const void* res, const float* slope2, const std::string& tg,
                          const Shortcut* sc = nullptr) -> bool {
      ConvFrameProblem fp;
      fp.A = in; fp.frames = nimg; fp.Hin = Hin; fp.Sin = Sin; fp.Pin = Sin * Sin; fp.Cin = Cin;
      fp.B = cu.w.w; fp.Cout = cu.cout; fp.ks = cu.ks; fp.stride = cu.stride;
      fp.Hout = Hout; fp.Sout = Hout; fp.Pout = Hout * Hout;
      fp.scale = cu.scale; fp.bias = cu.bias; fp.slope1 = slope1; fp.R = res; fp.slope2 = slope2; fp.C = out;
      if (sc != nullptr) {        // conv2 + shortcut conv in one GEMM: folded weights, scale 1, summed bias, then PReLU
        fp.B = sc->w->w; fp.scale = sc->ones; fp.bias = sc->bias;
        fp.A2 = sc->A2; fp.ds_Cin = sc->Cin; fp.ds_Sin = sc->Sin; fp.ds_Pin = sc->Sin * sc->Sin; fp.ds_stride = sc->stride;
      }
      void* table = b.alloc(conv_frame_table_bytes(fp));
      if (sizing) return true;
      ConvFramePlan* cp = new ConvFramePlan();
      plan->convframes.push_back(cp);
      if (conv_frame_plan(fp, cp) || conv_frame_bind_table(cp, table)) return false;
      double taps = 0;
      for (int oy = 0; oy < Hout; ++oy)
        for (int k = 0; k < cu.ks; ++k) {
          const int iy = oy * cu.stride + k - (cu.ks == 3 ? 1 : 0);
          taps += (iy >= 0 && iy < Hin) ? 1 : 0;
        }
      const double fl = 2.0 * (double)nimg * taps * taps * (double)Cin * (double)cu.cout +
                        (sc != nullptr ? 2.0 * (double)nimg * Hout * Hout * (double)sc->Cin * (double)cu.cout : 0.0);
      b.push(tg, [cp](cudaStream_t s) { return conv_frame_launch(*cp, s); }, fl);
      return true;
    };

    for (int b0 = 0; b0 < B; b0 += CB) {
      const int nb = std::min(CB, B - b0);
      const int nf = rg ? (int)N : nb * T;
      const long long f0 = rg ? 0 : (long long)b0 * T;
      // ---- stem: one fused kernel in bf16 mode (stem_fused.cu) ...
      if (!f32 && !train) {
        if (!sizing && b0 == 0 && stem_fused_plan(h->stem_wf.w, &plan->stemf)) return false;
        void* po = fb.pooled.data;
        const double fl = 2.0 * (double)nf * 1936.0 * 64.0 * 245.0;
        if (rg)
          b.push_direct("stem_fused", [=](cudaStream_t s) {
            return stem_fused_launch_ragged(pl->stemf, pl->args.video, pl->args.video_dt, pl->args.pitch,
                                            reinterpret_cast<const int4*>(pl->rag + pl->rag_items_off), pl->rag, pl->rag + 16,
                                            h->stem.scale, h->stem.bias, h->stem.slope, po, s);
          }, fl);
        else
          b.push_direct("stem_fused", [=](cudaStream_t s) {
            return stem_fused_launch(pl->stemf, pl->args.video, pl->args.video_dt, T, b0, nb, h->stem.scale, h->stem.bias,
                                     h->stem.slope, po, s);
          }, fl);
      } else
      // ---- ... else (kh,kw) patches -> GEMM over 5 temporal row-shift taps (+BN+PReLU) -> maxpool
      {
        void* col = fb.im2col;
        const int planes = P;
        b.push_direct("stem_patches", [=](cudaStream_t s) {
          return launch_stem_patches(pl->args.video, pl->args.video_dt, T, b0, nb, col, planes, s);
        });
        Epilogue ep = epilogue(fb.stem_out, 64, f32);
        ep.col_scale = h->stem.scale; ep.col_bias = h->stem.bias; ep.act = ACT_PRELU; ep.slope1 = h->stem.slope;
        const long long rows = (long long)nb * (T + 2) * 1936;       // tile rows include the gap frames
        // rows map 1:1 (TMA-store epilogue); rows of the gap frames hold don't-care values nobody reads
        std::vector<Tap> taps;
        for (int dt = 0; dt < 5; ++dt) taps.push_back(Tap{(dt - 2) * 1936, 0, dt * 64});
        // batch statistics over all frames of the batch, one chunk in training mode (gap frames of the clip-padded row
        // space excluded)
        if (!conv_bn(ep, h->stem, rows, (double)nf * 1936.0, (long long)(T + 2) * 1936, (long long)T * 1936, 0, 0,
                     [&](const Epilogue& e) { return b.gemm("stem_gemm", fb.im2col, rows, P * 64, h->stem.w, rows, taps, 1, 64, e); }))
          return false;
        void* so = fb.stem_out;
        void* po = fb.pooled.data;
        b.push("maxpool", [=](cudaStream_t s) { return launch_maxpool_stem(so, po, nf, T, f32 ? 1 : 0, s); });
        Act pv = fb.pooled; pv.rows = (long long)nf * 529;
        b.sync_op(pv);
      }
      // intermediate maps of this chunk, readable with avh_read_stage (no launch: a later chunk overwrites the entries,
      // so after a forward they hold the last chunk's frames)
      b.stage("stem", fb.pooled.data, act_dt, (long long)nf * 529 * 64);
      // ---- trunk
      Act cur = fb.pooled;
      for (int L = 0; L < 4; ++L) {
        const int Hn = HS[L], S = Hn + 1, Cc = 64 << L;
        for (int bi = 0; bi < 2; ++bi) {
          const BlockW& bw = h->blocks[L][bi];
          Act mid = fb.a[L][bi * 2], out = fb.a[L][bi * 2 + 1];
          mid.rows = out.rows = (long long)nf * S * S;
          {
            const long long n = (long long)nf * ((frame_mode && L > 0) ? Hn * Hn : S * S) * Cc;
            const std::string nm = "layer" + std::to_string(L + 1) + "." + std::to_string(bi);
            b.stage((nm + ".mid").c_str(), mid.data, act_dt, n);
            b.stage((nm + ".out").c_str(), out.data, act_dt, n);
            if (bw.has_ds && !frame_mode) b.stage((nm + ".ds").c_str(), fb.ds[L].data, act_dt, n);
          }
          const Act* res = &cur;
          Act dsout;
          if (frame_mode && L > 0) {
            const int Hp = bi == 0 ? HS[L - 1] : Hn, Sp = (bi == 0 && L == 1) ? Hp + 1 : Hp, Cin = bi == 0 ? Cc / 2 : Cc;
            if (!conv_frame(cur.op, Hp, Sp, Cin, bw.c1, mid.data, Hn, nf, bw.c1.slope, nullptr, nullptr,
                            (bi == 0 ? "conv_s2_c" : "conv3x3_c") + std::to_string(Cin)))
              return false;
            if (bw.has_ds) {
              // block 0 of layers 2-4: out = PReLU(BN2(conv2(mid)) + BN_ds(conv1x1_s2(x))) as ONE GEMM (the shortcut's
              // K steps read the block input x directly): no shortcut launch, no shortcut map written and re-read
              Shortcut sc;
              sc.A2 = cur.op; sc.Cin = Cin; sc.Sin = Sp; sc.stride = 2; sc.w = &bw.c2ds; sc.bias = bw.c2ds_bias; sc.ones = bw.ones;
              if (!conv_frame(mid.data, Hn, Hn, Cc, bw.c2, out.data, Hn, nf, bw.slope2, nullptr, nullptr,
                              "conv3x3_c" + std::to_string(Cc), &sc))
                return false;
            } else if (!conv_frame(mid.data, Hn, Hn, Cc, bw.c2, out.data, Hn, nf, nullptr, cur.data, bw.slope2,
                                   "conv3x3_c" + std::to_string(Cc)))
              return false;
            cur = out;
            continue;
          }
          if (bw.has_ds) {
            // stride-2: explicit im2col of the previous layer's padded map, conv1 and the 1x1 downsample read it
            const int Hp = HS[L - 1], Cin = Cc / 2;
            void* col = fb.col[L];
            const void* src = cur.op;
            const int CinP = Cin * P;
            b.push("im2col_s2", [=](cudaStream_t s) { return launch_im2col_s2(src, col, nf, Hp, Hp, CinP, s); });
            const long long rows = (long long)nf * Hn * Hn;
            std::vector<Tap> taps;
            for (int t = 0; t < 9; ++t) taps.push_back(Tap{0, t * CinP, t * Cin});
            Epilogue ep = epilogue(mid.data, Cc, f32);
            ep.col_scale = bw.c1.scale; ep.col_bias = bw.c1.bias; ep.act = ACT_PRELU; ep.slope1 = bw.c1.slope;
            ep.map_mode = MAP_2LEVEL; ep.S2 = Hn * Hn; ep.S1 = Hn; ep.H = Hn; ep.W = Hn;
            ep.O2 = S * S; ep.O1 = S; ep.O0 = 0;
            const std::string tag = "conv_s2_c" + std::to_string(Cin);
            const long long out_rows = (long long)nf * S * S;
            if (!conv_bn(ep, bw.c1, out_rows, (double)nf * Hn * Hn, 0, 0, S, Hn, [&](const Epilogue& e) {
                  return b.gemm(tag, col, rows, 9 * CinP, bw.c1.w, rows, taps, Cin / 64, Cin, e);
                }))
              return false;
            b.sync_op(mid);
            dsout = fb.ds[L];
            dsout.rows = mid.rows;
            Epilogue epd = epilogue(dsout.data, Cc, f32);
            epd.col_scale = bw.ds.scale; epd.col_bias = bw.ds.bias;
            epd.map_mode = MAP_2LEVEL; epd.S2 = Hn * Hn; epd.S1 = Hn; epd.H = Hn; epd.W = Hn;
            epd.O2 = S * S; epd.O1 = S; epd.O0 = 0;
            if (!conv_bn(epd, bw.ds, out_rows, (double)nf * Hn * Hn, 0, 0, S, Hn, [&](const Epilogue& e) {
                  return b.gemm("downsample", col, rows, 9 * CinP, bw.ds.w, rows, {Tap{0, 4 * CinP, 0}}, Cin / 64, Cin, e);
                }))
              return false;
            res = &dsout;
          } else {
            if (!conv3x3_s1(cur, bw.c1, mid, Hn, nf, bw.c1.slope, nullptr, nullptr)) return false;
          }
          if (!conv3x3_s1(mid, bw.c2, out, Hn, nf, nullptr, res, bw.slope2)) return false;
          cur = out;
        }
      }
      // ---- AdaptiveAvgPool2d(1) -> [nf, 512] rows f0.. of the ResEncoder output
      {
        const void* src = cur.data;
        char* dst = reinterpret_cast<char*>(pooled_feat.data) + (size_t)f0 * 512 * es;
        const int pitch = frame_mode ? 3 : 4;
        b.push("avgpool", [=](cudaStream_t s) { return launch_avgpool(src, dst, nf, 3, 3, 512, pitch, f32 ? 1 : 0, s); });
      }
    }
    b.sync_op(pooled_feat);
    // ---- SubModel.proj (hubert.py:321,327): Linear 512 -> D into the video columns of the fused buffer
    Epilogue ep = epilogue(reinterpret_cast<char*>(fused.data) + (size_t)v_off * es, E, f32);
    ep.col_bias = h->proj_v.bias;
    if (key.moddrop) b.cur_mod = 2;
    if (!b.linear("proj_video", pooled_feat.op, N, 512, h->proj_v.w, ep)) return false;
    // features_video = 0 * features_video (hubert.py:611-616): the ResNet still ran (its running statistics moved); add
    // fusion: the audio projection adds onto these zeros
    if (key.moddrop) b.zero_cols_on_drop(2, fused.data, N, E, v_off, D, es);
  }
  // ========================================================================== audio arm
  if (key.has_audio) {
    const int Fa = c.audio_feat_dim, Fp = round_up(Fa, 64);
    Act arows = b.act(N, Fp);       // zero-initialised; only the first Fa columns are ever written
    void* dst = arows.data;
    if (key.moddrop) b.cur_mod = 1;     // a dropped audio arm: its projection is skipped
    if (rg)
      b.push_direct("audio_rows", [=](cudaStream_t s) {
        return launch_bct_to_rows_ragged(pl->args.audio, pl->args.audio_dt, pl->args.as[0], pl->args.as[1], pl->args.as[2],
                                         B, Fa, pl->rag + 16, dst, act_dt, Fp, N, s);
      });
    else
      b.push_direct("audio_rows", [=](cudaStream_t s) {
        return launch_bct_to_rows(pl->args.audio, pl->args.audio_dt, pl->args.as[0], pl->args.as[1], pl->args.as[2],
                                  B, Fa, T, dst, act_dt, Fp, s);
      });
    b.sync_op(arows);
    Epilogue ep = epilogue(reinterpret_cast<char*>(fused.data) + (size_t)a_off * es, E, f32);
    ep.col_bias = h->proj_a.bias;
    if (c.modality_fuse == AVH_FUSE_ADD && key.has_video) {     // features_audio + features_video
      ep.R = ep.C; ep.ldr = E; ep.r_fp32 = f32 ? 1 : 0;
    }
    if (!b.linear("proj_audio", arows.op, N, Fp, h->proj_a.w, ep)) return false;
    b.cur_mod = 0;
    // features_audio = 0 * features_audio: with add fusion the skipped projection leaves the video features alone
    if (key.moddrop && c.modality_fuse == AVH_FUSE_CONCAT) b.zero_cols_on_drop(1, fused.data, N, E, a_off, D, es);
  }
  // a missing modality contributes zeros [B,D,T] (hubert.py:703-708): with concat its columns stay at the
  // arena's zero fill (nothing ever writes them for this plan); with add there is nothing to add.

  // ========================================================================== fusion LN + post_extract_proj
  float* x = b.f32buf(N * D);      // residual stream, fp32
  if (enc_only) {
    // TransformerEncoder.forward on the caller's features: x = features with padded frames zeroed (wav2vec2.py:869-870)
    b.push_direct("load_features", [=](cudaStream_t s) {
      return launch_load_rows(pl->args.xin, pl->args.xin_dt, x, hm ? pl->mask_dev : nullptr, N, D, s);
    });
  } else {
    b.stage("fused", fused.data, act_dt, N * E);     // pre-LayerNorm features (features_pen)
    if (!sizing) { plan->fused_buf = fused.data; plan->fused_dt = act_dt; }
    Act lnE = b.act(N, E);
    if (h->has_post_proj) {
      b.layernorm("fuse_ln", fused.data, act_dt, h->fuse_ln_g, h->fuse_ln_b, 1e-5f, lnE);
      b.stage("fused_ln", lnE.data, act_dt, N * E);
      Epilogue ep = epilogue(x, D, true);
      ep.col_bias = h->post_proj.bias;
      ep.row_zero = hm ? plan->mask_dev : nullptr;      // index_put(x, padding_mask, 0), wav2vec2.py:869-870
      if (!b.linear("post_extract_proj", lnE.op, N, E, h->post_proj.w, ep)) return false;
    } else {
      // no post_extract_proj (embed == D): the LN output is the encoder input; zero padded rows here
      const void* src = fused.data;
      float* g = h->fuse_ln_g; float* be = h->fuse_ln_b;
      b.push("fuse_ln", [=](cudaStream_t s) {
        return launch_layernorm(src, act_dt, E, g, be, 1e-5f, x, nullptr, DT_BF16, hm ? pl->mask_dev : nullptr, N, E, s);
      });
      b.stage("fused_ln", x, DT_F32, N * E);
    }
  }
  if (train) {      // features = self.dropout_input(features), hubert.py:729
    b.push("dropout", [=](cudaStream_t s) {
      return pl->p_in > 0.f ? launch_dropout(x, DT_F32, nullptr, N * D, pl->p_in, pl->seed, 1u, s) : 0;
    });
  }
  if (c.capture_stages) {      // x is overwritten in place by the encoder: keep a copy for stage-level tests
    float* enc_in_copy = b.f32buf(N * D);
    b.push("stage_copy", [=](cudaStream_t s) {
      return cudaMemcpyAsync(enc_in_copy, x, (size_t)N * D * 4, cudaMemcpyDeviceToDevice, s) == cudaSuccess ? 0 : 1;
    });
    b.stage("enc_in", enc_in_copy, DT_F32, N * D);
  }

  // ========================================================================== positional conv + GELU + residual
  {
    const int G = 64, Tp = T + G;
    const long long pad_rows = rg ? N + (long long)G * B : (long long)B * Tp;
    void* xpad = b.alloc((size_t)pad_rows * P * D * 2);      // bf16 [B*(T+64), P*D], gap rows stay zero
    const int planes = P;
    int* row_map = nullptr;
    if (rg) {
      // packed clips: clip b at padded rows [cu[b] + 64 b, +T_b); the kernel also zeroes the gap rows (they move from
      // call to call) and writes the padded-row -> packed-row map the convolution's epilogue stores through
      row_map = reinterpret_cast<int*>(b.alloc((size_t)pad_rows * 4));
      if (!sizing) plan->pos_row_map = row_map;
      b.push("pos_pad", [=](cudaStream_t s) { return launch_pos_pad_ragged(x, D, xpad, row_map, pl->rag + 16, B, D, G, pad_rows, s); });
    } else
    b.push("pos_pad", [=](cudaStream_t s) { return launch_split_rows(x, D, xpad, planes, N, D, T, Tp, s); });
    const int KT = c.conv_pos, win = h->pos_window;
    std::vector<Tap> taps;
    for (int k = 0; k < KT; ++k) taps.push_back(Tap{k - KT / 2, 0, k * win});
    Epilogue ep = epilogue(x, D, true);
    ep.col_bias = h->pos_bias; ep.act = ACT_GELU;
    ep.R = x; ep.ldr = D; ep.r_fp32 = 1;
    if (rg) ep.row_map = row_map;
    else { ep.map_mode = MAP_2LEVEL; ep.S2 = Tp; ep.S1 = Tp; ep.H = 1; ep.W = T; ep.O2 = T; ep.O1 = 0; ep.O0 = 0; }
    if (!b.gemm("pos_conv", xpad, pad_rows, P * D, h->pos_w, pad_rows, taps, win / 64, D, ep, 64, h->pos_acol))
      return false;
  }

  // ========================================================================== transformer layers
  float* dtmp = train ? b.f32buf(N * D) : nullptr;     // block output before dropout + add
  Act hbuf = b.act(N, D);          // LayerNorm output / post-LN operand copy of x
  Act qkv = b.act(N, 3 * D);
  Act ctx = b.act(N, D);
  Act ffn = b.act(N, F);
  float* tmp = c.layer_norm_first ? nullptr : b.f32buf(N * D);

  // post-LN: x = LayerNorm(src) in place of the residual stream (src = x or tmp)
  auto post_ln = [&](const float* src, const float* g, const float* be) {
    b.push("layer_ln", [=](cudaStream_t s) { return launch_layernorm(src, DT_F32, D, g, be, 1e-5f, x, nullptr, DT_BF16, nullptr, N, D, s); });
  };
  if (!c.layer_norm_first) {
    // encoder-level LayerNorm right after the positional conv (wav2vec2.py:876-877)
    post_ln(x, h->enc_ln_g, h->enc_ln_b);
    if (!train) b.split(x, D, hbuf.op, N, D);      // operand copy of the residual stream (post-LN blocks read x itself)
  }
  if (train) {      // x = F.dropout(x, p=self.dropout, training=self.training), wav2vec2.py:879
    b.push("dropout", [=](cudaStream_t s) {
      return pl->p_enc > 0.f ? launch_dropout(x, DT_F32, nullptr, N * D, pl->p_enc, pl->seed, 2u, s) : 0;
    });
    if (!c.layer_norm_first) b.split(x, D, hbuf.op, N, D);
  }
  const int n_layers = key.output_layer > 0 ? std::min(key.output_layer, c.encoder_layers) : c.encoder_layers;
  // measured (tools/att_bench.py, Large head count): tcgen05 11.4 vs 12.8 us at 16 x 150, 21.6 vs 29.0 at 8 x 300,
  // 31.9 vs 44.3 at 4 x 600; short clips (64 x 38 frames: 12.6 vs 9.3 us) stay on the mma.sync kernel
  const bool att_tc = !f32 && (rg || T > 96) && (size_t)((T + 127) / 128 * 128) * 4 <= 48 * 1024;
  for (int l = 0; l < n_layers; ++l) {
    const LayerW& lw = h->layers[l];
    b.cur_layer = l;               // LayerDrop (training mode) skips every launch of a dropped layer
    if (c.layer_norm_first) b.layernorm("layer_ln", x, DT_F32, lw.ln1_g, lw.ln1_b, 1e-5f, hbuf);
    {   // fused QKV projection
      Epilogue ep = epilogue(qkv.data, 3 * D, f32);
      ep.col_bias = lw.qkv.bias;
      if (!b.linear("qkv_proj", hbuf.op, N, D, lw.qkv.w, ep)) return false;
    }
    {
      const void* q = qkv.data; void* o = ctx.data;
      const double att_flops = 4.0 * (double)B * Hh * (double)T * (double)T * 64.0;   // QK^T + PV, dense (padding not excluded)
      if (att_tc) {
        // bf16 mode: tcgen05 / TMEM kernel (attention_tc.cu)
        if (!sizing && l == 0 && attention_tc_plan(q, N, B, T, D, Hh, &plan->att)) return false;
        b.push("attention", [=](cudaStream_t s) {
          return attention_tc_launch(pl->att, hm ? pl->mask_dev : nullptr, rg ? pl->rag + 16 : nullptr, o, s);
        }, att_flops);
      } else {
        b.push("attention", [=](cudaStream_t s) {
          return launch_attention(q, hm ? pl->mask_dev : nullptr, o, B, T, D, Hh, f32 ? 1 : 0, s);
        }, att_flops);
      }
      b.sync_op(ctx);
    }
    // training mode: block output -> dtmp, then target (+)= dropout(dtmp) (dropout1 / dropout3, wav2vec2.py:980,990);
    // with p = 0 this is the eval arithmetic (fp32 block output added to the fp32 residual stream)
    auto dropout_add = [&](unsigned site) {
      float* target = c.layer_norm_first ? x : tmp;
      if (!c.layer_norm_first)
        b.push("dropout", [=](cudaStream_t s) {
          return cudaMemcpyAsync(tmp, x, (size_t)N * D * 4, cudaMemcpyDeviceToDevice, s) == cudaSuccess ? 0 : 1;
        });
      b.push("dropout", [=](cudaStream_t s) { return launch_dropout(target, DT_F32, dtmp, N * D, pl->p_enc, pl->seed, site, s); });
    };
    {   // out_proj + residual
      Epilogue ep = epilogue(c.layer_norm_first ? x : tmp, D, true);
      ep.col_bias = lw.out.bias; ep.R = x; ep.ldr = D; ep.r_fp32 = 1;
      if (train) { ep.C = dtmp; ep.R = nullptr; }
      if (!b.linear("out_proj", ctx.op, N, D, lw.out.w, ep)) return false;
      if (train) dropout_add(16u + 4u * (unsigned)l);
    }
    if (c.layer_norm_first) b.layernorm("layer_ln", x, DT_F32, lw.ln2_g, lw.ln2_b, 1e-5f, hbuf);
    else {
      post_ln(tmp, lw.ln1_g, lw.ln1_b);
      b.split(x, D, hbuf.op, N, D);
    }
    {   // fc1 + GELU (erf form, fp32: fairseq/fairseq/modules/gelu.py:95-96)
      Epilogue ep = epilogue(ffn.data, F, f32);
      ep.col_bias = lw.fc1.bias; ep.act = ACT_GELU;
      if (!b.linear("fc1", hbuf.op, N, D, lw.fc1.w, ep)) return false;
      if (train) {      // dropout2 = activation_dropout after the GELU, wav2vec2.py:987
        void* fd = ffn.data;
        const unsigned site = 17u + 4u * (unsigned)l;
        b.push("dropout", [=](cudaStream_t s) {
          return pl->p_act > 0.f ? launch_dropout(fd, act_dt, nullptr, N * F, pl->p_act, pl->seed, site, s) : 0;
        });
      }
      b.sync_op(ffn);
    }
    {   // fc2 + residual
      Epilogue ep = epilogue(c.layer_norm_first ? x : tmp, D, true);
      ep.col_bias = lw.fc2.bias; ep.R = x; ep.ldr = D; ep.r_fp32 = 1;
      if (train) { ep.C = dtmp; ep.R = nullptr; }
      if (!b.linear("fc2", ffn.op, N, F, lw.fc2.w, ep)) return false;
      if (train) dropout_add(18u + 4u * (unsigned)l);
    }
    if (!c.layer_norm_first) {
      post_ln(tmp, lw.ln2_g, lw.ln2_b);
      if (l + 1 < n_layers) b.split(x, D, hbuf.op, N, D);
    }
  }
  b.cur_layer = -1;
  // ========================================================================== output
  const bool final_ln = c.layer_norm_first && key.output_layer == 0;
  float* g = h->enc_ln_g; float* be = h->enc_ln_b;
  if (rg) {
    // packed rows -> the caller's [B, pitch_T, D] tensor, zeros at the pad positions
    float* y = x;
    if (final_ln) {
      y = b.f32buf(N * D);
      b.push("final_ln", [=](cudaStream_t s) { return launch_layernorm(x, DT_F32, D, g, be, 1e-5f, y, nullptr, DT_BF16, nullptr, N, D, s); });
    }
    b.push_direct("unpack", [=](cudaStream_t s) {
      return launch_unpack_rows(y, pl->rag + 16, pl->args.out, pl->args.out_dt, B, pl->args.pitch, D, s);
    });
  } else if (final_ln) {
    b.push_direct("final_ln", [=](cudaStream_t s) {
      return launch_layernorm(x, DT_F32, D, g, be, 1e-5f, nullptr, pl->args.out, pl->args.out_dt, nullptr, N, D, s);
    });
  } else {
    b.push_direct("final_ln", [=](cudaStream_t s) { return launch_convert(x, DT_F32, pl->args.out, pl->args.out_dt, N * D, s); });
  }
  if (bytes_out) *bytes_out = b.sizer.used;
  return true;
}

// ============================================================================ encoder training plan
// TransformerEncoder forward with saved activations + its backward, pre-LN or post-LN layers.  Pre-LN forward:
// x0 = index_put(features, mask, 0); c = pos_conv(x0) + b; x1 = m2 (x0 + GELU(c)); per layer h1 = LN1(x);
// qkv = h1 Wqkv^T + b; ctx = Attn(qkv) (+ log-sum-exp per row); xm = x + m(16+4l) (ctx Wo^T + bo); h2 = LN2(xm);
// u = h2 W1^T + b1; g = m(17+4l) GELU(u); x' = xm + m(18+4l) (g W2^T + b2); y = LN(x_L).
// Post-LN forward (wav2vec2.py:872-879, 993-1012): s = x0 + GELU(c); x1 = m2 LN(s); per layer qkv = x Wqkv^T + b (h1 = x);
// r1 = x + m(16+4l) (ctx Wo^T + bo); y1 = LN1(r1) (h2 = y1); r2 = y1 + m(18+4l) (g W2^T + b2); x' = LN2(r2); y = x_L
// (no final LayerNorm; encoder.layer_norm is the one after the positional conv and keeps its gradient slot).  Its
// backward: dr2 = LN2^T(dx; r2), dr1 = LN1^T(dr2 + dL/dy1; r1), dx = dr1 + dL/dx through qkv, ds = LN^T(m2 dx1; s), each
// LayerNorm backward also writing the masked gradient of the block that feeds it (launch_ln_post_bwd).
// Tail modes: x0 = m1 post_extract_proj(LN(fused)) before the zeroing.
// m_site = the dropout mask of that site (philox.cuh, p = key.p_in for site 1, p_act for 17+4l, p_enc otherwise; a
// site with p = 0 is no mask and no launch).  A layer dropped by LayerDrop is the identity: its steps are skipped, an
// on-drop step copies x into x' and zeroes the layer's gradients.  Backward: the chain rule of exactly that graph —
// every contraction on the tcgen05 GEMM (dX = dY W with W^T packed at finalisation; dW = dY^T X with both operands
// transposed by transpose_split, K = tokens), the rest in backward_ops.cu / train_dropout.cu, every mask regenerated
// from (seed, site, element).
// Gradient layout (fp32, `grad_floats` values), in this order — the Python mirror walks the same list:
//   per layer l: [q,k,v]_proj.weight (3 x [D,D], contiguous), [q,k,v]_proj.bias (3 x [D]), out_proj.weight [D,D],
//   out_proj.bias [D], self_attn_layer_norm.{weight,bias}, fc1.weight [F,D], fc1.bias [F], fc2.weight [D,F], fc2.bias [D],
//   final_layer_norm.{weight,bias};  then encoder.layer_norm.{weight,bias};  then pos_conv.0.bias [D],
//   pos_conv.0.weight_g [KT], pos_conv.0.weight_v [D, D/G, KT].
long long enc_layer_grad_floats(int D, int F) { return 4ll * D * D + 4ll * D + 2ll * D + 2ll * D * F + F + D + 2ll * D; }
long long frontend_grad_floats(const avh_config& c, bool has_video, bool has_audio);
long long enc_grad_floats(const avh_config& c, int tail = 0, bool has_video = true, bool has_audio = true) {
  const int D = c.encoder_embed_dim, F = c.encoder_ffn_embed_dim;
  const int E = c.modality_fuse == AVH_FUSE_CONCAT ? 2 * D : D;
  long long n = c.encoder_layers * enc_layer_grad_floats(D, F) + 2ll * D + D + c.conv_pos +
                (long long)D * (D / c.conv_pos_groups) * c.conv_pos;
  if (tail) n += (E != D ? (long long)D * E + D : 0) + 2ll * E;      // post_extract_proj.{weight,bias}, layer_norm.{weight,bias}
  if (tail == 2) n += frontend_grad_floats(c, has_video, has_audio);
  return n;
}

// Weight gradients of the grouped positional convolution + weight-norm backward (wav2vec2.py:822-834):
// dw[o, i, k] = sum_{b,t} dc[b,t,o] x0[b, t + k - KT/2, g(o) cg + i].  Per group one GEMM over K = the zero-gapped token
// axis: A = rows [g cg, +cg) of dc^T, B = the (tap, input channel) rows of the group — shifted copies of x0^T — so that
// N = KT cg; output [cg, KT cg] = dw of the group as (o, tap, in).  Then dg, dv of w = g v / ||v||.
bool posconv_wgrad(Builder& b, avh_handle* h, const float* dc, const float* x0, long long N, int B, int T, float* g_wg,
                   float* g_wv) {
  const avh_config& c = h->cfg;
  const int D = c.encoder_embed_dim, KT = c.conv_pos, G = c.conv_pos_groups, cg = D / G, P = b.P;
  const int Tp = T + 64;
  const long long kp = ((long long)B * Tp + 63) / 64 * 64;
  void* dcT = b.alloc((size_t)D * P * kp * 2);
  void* x0T = b.alloc((size_t)D * P * kp * 2);
  void* XS = b.alloc((size_t)KT * cg * P * kp * 2);
  float* dw = b.f32buf((long long)D * KT * cg);
  float* norms = b.f32buf(KT);
  const int planes = P;
  b.push("transpose", [=](cudaStream_t s) { return launch_transpose_split(dc, DT_F32, D, N, D, dcT, planes, kp, 1.0f, s, T, Tp); });
  b.push("transpose", [=](cudaStream_t s) { return launch_transpose_split(x0, DT_F32, D, N, D, x0T, planes, kp, 1.0f, s, T, Tp); });
  for (int g = 0; g < G; ++g) {
    b.push("pos_conv_shift", [=](cudaStream_t s) { return launch_posconv_shift(x0T, XS, g, cg, KT, planes, kp, s); });
    PackedW xw;
    xw.w = reinterpret_cast<bf16*>(XS); xw.n = KT * cg; xw.k = (int)kp; xw.kpad = (int)kp;
    const Epilogue ep = epilogue(dw + (size_t)g * cg * KT * cg, (long long)KT * cg, true);
    const char* a = reinterpret_cast<const char*>(dcT) + (size_t)g * cg * P * kp * 2;
    if (!b.linear("pos_conv_wgrad", a, cg, (int)kp, xw, ep)) return false;
  }
  const float* v = h->pos_v_raw; const float* gg = h->pos_g_raw;
  b.push("weight_norm_bwd", [=](cudaStream_t s) { return launch_posconv_weightnorm_bwd(dw, v, gg, D, cg, KT, g_wg, g_wv, norms, s); });
  return true;
}

// Gradients of the feature extractors (mode 2), after the tail's: feature_extractor_audio.proj.{weight [D, Fp], bias}
// (Fp = audio_feat_dim rounded up to 64, the columns past audio_feat_dim are zero), feature_extractor_video.proj.{weight
// [D,512], bias}, then the ResNet: frontend3D.0.weight as [64, 5, 64] (dt, kh*7+kw padded to 64), frontend3D.1.{weight,bias},
// frontend3D.2.weight; per BasicBlock conv1.weight [C, 3,3,Cin] (tap-major, channel-minor), bn1.{weight,bias},
// relu1.weight, conv2.weight, bn2.{weight,bias}, relu2.weight, and for the first block of layers 2-4 downsample.0.weight
// [C, Cin], downsample.1.{weight,bias}.  The Python mirror permutes the conv weights back to [C, Cin, kh, kw].
long long frontend_grad_floats(const avh_config& c, bool has_video, bool has_audio) {
  const int D = c.encoder_embed_dim;
  long long n = 0;
  if (has_audio) n += (long long)D * round_up(c.audio_feat_dim, 64) + D;
  if (has_video) {
    n += (long long)D * 512 + D + 64 * 320 + 3 * 64;
    int cin = 64;
    for (int L = 0; L < 4; ++L) {
      const int C = 64 << L;
      for (int bi = 0; bi < 2; ++bi) {
        n += (long long)C * 9 * cin + 3 * C + (long long)C * 9 * C + 3 * C;
        if (L > 0 && bi == 0) n += (long long)C * cin + 2 * C;
        cin = C;
      }
    }
  }
  return n;
}

bool build_encoder_train_plan(avh_handle* h, Plan* plan, bool sizing, size_t* bytes_out) {
  Builder b(h, plan, sizing);
  const avh_config& c = h->cfg;
  const PlanKey& key = plan->key;
  const int P = b.P;
  const bool f32 = b.f32;
  const int B = key.B, T = key.T, D = c.encoder_embed_dim, F = c.encoder_ffn_embed_dim, Hh = c.encoder_attention_heads;
  const int L = c.encoder_layers;
  const long long N = (long long)B * T;
  const long long Kp = (N + 63) / 64 * 64;                  // token count padded to whole K blocks (wgrad GEMMs)
  const size_t es = b.es;
  const int act_dt = b.act_dt;
  Plan* pl = plan;
  const bool post = !c.layer_norm_first;
  {
    unsigned char* md = b.mask_buf(N);
    if (!sizing) plan->mask_dev = md;
  }
  const bool hm = key.has_mask;
  const int tail = key.kind == PlanKind::FullTrain ? 2 : (key.kind == PlanKind::TailTrain ? 1 : 0);
  const bool full = tail == 2;
  const float p_in = key.p_in, p_enc = key.p_enc, p_act = key.p_act;
  const bool ldrop = key.layerdrop;
  unsigned long long* seed = key.dropout() ? reinterpret_cast<unsigned long long*>(b.alloc(16)) : nullptr;
  if (!sizing) plan->seed_dev = seed;
  float* dtmp = p_enc > 0.f ? b.f32buf(N * D) : nullptr;     // block output before dropout + residual; backward: m * dx
  // stream-K workspace for the lip ResNet's weight-gradient GEMMs (a handful of output tiles, K = pixels)
  if (!f32 && full) b.stream_k_workspace();
  const int E = c.modality_fuse == AVH_FUSE_CONCAT ? 2 * D : D;
  const long long GF = enc_grad_floats(c, tail, key.has_video, key.has_audio);
  float* grads = b.f32buf(GF);
  float* dy = b.f32buf(N * D);
  float* dxo = b.f32buf(N * D);
  if (!sizing) { plan->grads = grads; plan->grad_floats = GF; plan->dy_in = dy; plan->dx_out = dxo; }
  // gradient bucket [begin, end) of the flat buffer is final here: a direct (never captured) step hands it to the caller —
  // converted into the caller's buffer when avh_encoder_backward_buckets runs the plan — and records the bucket's event,
  // so that an all-reduce on another stream can start while the rest of the backward still runs
  auto grad_mark = [&](long long begin, long long end) {
    if (end <= begin) return;
    int k = -1;
    if (!sizing) {
      Plan::GradBucket gb{begin, end, nullptr};
      cudaEventCreateWithFlags(&gb.ev, cudaEventDisableTiming);
      plan->buckets.push_back(gb);
      k = (int)plan->buckets.size() - 1;
    }
    b.push_direct("grad_bucket", [=](cudaStream_t s) {
      const CallArgs& a = pl->args;
      if (a.grads_out == nullptr) return 0;
      const Plan::GradBucket& gb = pl->buckets[k];
      const size_t es = a.grads_dt == DT_F32 ? 4 : 2;
      if (launch_convert(pl->grads + gb.begin, DT_F32, reinterpret_cast<char*>(a.grads_out) + (size_t)gb.begin * es, a.grads_dt,
                         gb.end - gb.begin, s))
        return 1;
      return cudaEventRecord(gb.ev, s) == cudaSuccess ? 0 : 1;
    });
  };

  // ---------------------------------------------------------------- saved activations
  float* x0 = b.f32buf(N * D);
  float* cpre = b.f32buf(N * D);                               // positional conv output before the GELU
  std::vector<float*> xin(L + 1), xmid(L);
  std::vector<Act> h1(L), qkv(L), ctx(L), h2(L), u(L), g(L);
  std::vector<float*> lse(L);
  for (int l = 0; l <= L; ++l) xin[l] = b.f32buf(N * D);
  // post-LN: h1 = x_l itself, h2 = y1 = LN1(r1) (both also the residual stream, fp32); r2 = y1 + block before LN2;
  // spre = x0 + GELU(c) before the encoder LayerNorm
  std::vector<float*> y1(post ? L : 0), r2(post ? L : 0);
  float* spre = post ? b.f32buf(N * D) : nullptr;
  // fp32 residual-stream tensor as a GEMM input: fp32 mode reads the tensor itself, bf16 mode a bf16 copy
  auto stream_act = [&](float* v) {
    Act a;
    a.rows = N; a.C = D;
    a.data = f32 ? v : b.alloc((size_t)N * D * 2);
    a.op = f32 ? b.alloc((size_t)N * D * 2 * P) : a.data;
    return a;
  };
  for (int l = 0; l < L; ++l) {
    xmid[l] = b.f32buf(N * D);
    if (post) {
      y1[l] = b.f32buf(N * D); r2[l] = b.f32buf(N * D);
      h1[l] = stream_act(xin[l]); h2[l] = stream_act(y1[l]);
      qkv[l] = b.act(N, 3 * D); ctx[l] = b.act(N, D);
    } else {
      h1[l] = b.act(N, D); qkv[l] = b.act(N, 3 * D); ctx[l] = b.act(N, D); h2[l] = b.act(N, D);
    }
    u[l] = b.act(N, F); g[l] = b.act(N, F);
    lse[l] = b.f32buf((long long)B * Hh * T);
  }

  // ================================================================ forward
  float* fused = nullptr;                 // tail: the caller's fused features [N, E] (fp32 copy) and their LayerNorm
  Act fln;
  // ---- mode 2: the feature extractors inside the plan, every convolution as explicit patches -> GEMM on dense NHWC maps
  struct ConvSave {                      // what the backward of one conv + BatchNorm (+ residual) (+ PReLU) needs
    const ConvUnit* cu = nullptr;
    Act in, raw, res, out;               // input map, raw conv output, residual added after the BatchNorm, block output
    int H = 0, Ho = 0, pad = 0;
    float* stat = nullptr;               // batch mean | rstd
    const float* slope = nullptr;        // PReLU after (BatchNorm + residual), or null
  };
  std::vector<ConvSave> convs;           // forward order: stem, then per block conv1, [downsample], conv2
  Act feat, arows, act0, p0;
  const long long nfr = N;               // frames
  void* colbuf = nullptr;
  void* stemcol = nullptr;
  unsigned char* pool_arg = nullptr;     // bf16 mode: window position of every max-pool maximum
  double* bn_sums = nullptr;
  float *bn_scale = nullptr, *bn_bias = nullptr;
  const int v_off = c.modality_fuse == AVH_FUSE_CONCAT ? D : 0;
  const int Fa = c.audio_feat_dim, Fp = round_up(Fa > 0 ? Fa : 64, 64);
  if (full) {
    fused = b.f32buf(N * E);
    fln = b.act(N, E);
    bn_sums = reinterpret_cast<double*>(b.alloc((size_t)BN_SLOTS * 3 * 512 * sizeof(double)));
    bn_scale = b.f32buf(512); bn_bias = b.f32buf(512);
    if (key.has_video) {
      colbuf = b.alloc((size_t)nfr * 484 * 576 * P * 2);
      stemcol = b.alloc((size_t)nfr * 1936 * 320 * P * 2);      // stem patches: kept for the weight gradient
      if (!f32) pool_arg = reinterpret_cast<unsigned char*>(b.alloc((size_t)nfr * 484 * 64));
      auto bn_fwd = [&](ConvSave& cs, long long rows, const float* slope1, const Act* res, const float* slope2, const Act& out) {
        const ConvUnit* cu = cs.cu;
        const int Cc = cu->cout;
        const void* rawp = cs.raw.data; void* outp = out.data;
        const void* resp = res ? res->data : nullptr;
        const float *gm = cu->gamma, *bt = cu->beta;
        float *rm = cu->rmean, *rv = cu->rvar;
        float* st = b.f32buf(2 * Cc);
        cs.stat = st; cs.out = out; cs.slope = slope1 ? slope1 : slope2;
        if (res) cs.res = *res;
        b.push("bn_train", [=](cudaStream_t s) { return launch_bn_stats(rawp, act_dt, rows, Cc, 0, 0, 0, 0, bn_sums, s); });
        b.push("bn_train", [=](cudaStream_t s) {
          return launch_bn_finalize(bn_sums, (double)rows, gm, bt, 1e-5f, pl->bn_momentum, rm, rv, bn_scale, bn_bias, Cc, s);
        });
        b.push("bn_train", [=](cudaStream_t s) { return launch_bn_stat_from_affine(bn_scale, bn_bias, gm, bt, Cc, st, s); });
        b.push("bn_train", [=](cudaStream_t s) {
          return launch_bn_apply(rawp, outp, act_dt, rows, Cc, bn_scale, bn_bias, slope1, resp, slope2, 0, 0, s);
        });
        b.sync_op(out);
      };
      auto conv_fwd = [&](const ConvUnit& cu, const Act& in, int H, int pad, ConvSave* cs) -> bool {
        const int Ho = (H + 2 * pad - cu.ks) / cu.stride + 1;
        const int K = cu.ks * cu.ks * cu.cin;
        const long long rows = nfr * Ho * Ho;
        cs->cu = &cu; cs->in = in; cs->H = H; cs->Ho = Ho; cs->pad = pad;
        cs->raw = b.act(rows, cu.cout);
        const void* xin = in.data;
        const int planes = P, ks = cu.ks, st = cu.stride, cin = cu.cin;
        b.push("im2col", [=](cudaStream_t s) { return launch_im2col2d(xin, act_dt, nfr, H, cin, ks, st, pad, Ho, colbuf, planes, s); });
        return b.linear("conv_gemm", colbuf, rows, K, cu.w, epilogue(cs->raw.data, cu.cout, f32));
      };
      // stem: Conv3d as patches [frames * 1936, 5 * 64] x the packed stem weights
      {
        ConvSave cs;
        cs.cu = &h->stem; cs.H = 88; cs.Ho = 44;
        const long long rows = nfr * 1936;
        cs.raw = b.act(rows, 64);
        const int planes = P;
        b.push_direct("stem_patches", [=](cudaStream_t s) {
          return launch_im2col_stem(pl->args.video, pl->args.video_dt, B, T, stemcol, planes, s);
        });
        // K = dt*64 + kh*8 + kw
        if (!b.linear("stem_gemm", stemcol, rows, 320, h->stem_wf, epilogue(cs.raw.data, 64, f32))) return false;
        act0 = b.act(rows, 64);
        bn_fwd(cs, rows, h->stem.slope, nullptr, nullptr, act0);
        convs.push_back(cs);
        p0 = b.act(nfr * 484, 64);
        const void* a0 = act0.data; void* pp = p0.data;
        b.push("maxpool", [=](cudaStream_t s) { return launch_maxpool_dense(a0, pp, act_dt, nfr, 44, 64, 22, s, pool_arg); });
        b.sync_op(p0);
      }
      Act cur = p0;
      int H = 22;
      for (int L = 0; L < 4; ++L)
        for (int bi = 0; bi < 2; ++bi) {
          const BlockW& bw = h->blocks[L][bi];
          ConvSave c1, c2, cd;
          if (!conv_fwd(bw.c1, cur, H, 1, &c1)) return false;
          const int Ho = c1.Ho, Cc = bw.c1.cout;
          const long long rows = nfr * Ho * Ho;
          Act a1 = b.act(rows, Cc);
          bn_fwd(c1, rows, bw.c1.slope, nullptr, nullptr, a1);
          convs.push_back(c1);
          Act resid = cur;
          if (bw.has_ds) {
            if (!conv_fwd(bw.ds, cur, H, 0, &cd)) return false;
            Act dso = b.act(rows, Cc);
            bn_fwd(cd, rows, nullptr, nullptr, nullptr, dso);
            convs.push_back(cd);
            resid = dso;
          }
          if (!conv_fwd(bw.c2, a1, Ho, 1, &c2)) return false;
          Act outb = b.act(rows, Cc);
          bn_fwd(c2, rows, nullptr, &resid, bw.slope2, outb);
          convs.push_back(c2);
          cur = outb;
          H = Ho;
        }
      feat = b.act(N, 512);
      b.stage("resnet", feat.data, act_dt, N * 512);
      {
        const void* src = cur.data; void* dst = feat.data;
        b.push("avgpool", [=](cudaStream_t s) { return launch_avgpool_dense(src, dst, act_dt, nfr, 9, 512, s); });
        b.sync_op(feat);
      }
      Epilogue ep = epilogue(fused + v_off, E, true);
      ep.col_bias = h->proj_v.bias;
      if (key.moddrop) b.cur_mod = 2;      // modality dropout as in the training-mode forward (build_plan)
      if (!b.linear("proj_video", feat.op, N, 512, h->proj_v.w, ep)) return false;
      if (key.moddrop) b.zero_cols_on_drop(2, fused, N, E, v_off, D, 4);
    }
    if (key.has_audio) {
      arows = b.act(N, Fp);
      void* dst = arows.data;
      if (key.moddrop) b.cur_mod = 1;
      b.push_direct("audio_rows", [=](cudaStream_t s) {
        return launch_bct_to_rows(pl->args.audio, pl->args.audio_dt, pl->args.as[0], pl->args.as[1], pl->args.as[2], B, Fa, T, dst,
                                  act_dt, Fp, s);
      });
      b.sync_op(arows);
      Epilogue ep = epilogue(fused, E, true);
      ep.col_bias = h->proj_a.bias;
      if (c.modality_fuse == AVH_FUSE_ADD && key.has_video) { ep.R = ep.C; ep.ldr = E; ep.r_fp32 = 1; }
      if (!b.linear("proj_audio", arows.op, N, Fp, h->proj_a.w, ep)) return false;
      b.cur_mod = 0;
      if (key.moddrop && c.modality_fuse == AVH_FUSE_CONCAT) b.zero_cols_on_drop(1, fused, N, E, 0, D, 4);
    }
  }
  if (tail) {
    // AVHubertModel.extract_finetune after the feature extractors: features = layer_norm(fused);
    // features = post_extract_proj(features) (concat fusion); index_put(padded frames, 0)   (hubert.py:719-727, wav2vec2.py:869)
    if (!full) {
      fused = b.f32buf(N * E);
      fln = b.act(N, E);
      b.push_direct("load_features", [=](cudaStream_t s) {
        return launch_load_rows(pl->args.xin, pl->args.xin_dt, fused, nullptr, N, E, s);
      });
    }
    if (!sizing) { plan->fused_buf = fused; plan->fused_dt = DT_F32; }
    if (h->has_post_proj) {
      b.layernorm("fuse_ln", fused, DT_F32, h->fuse_ln_g, h->fuse_ln_b, 1e-5f, fln);
      Epilogue ep = epilogue(x0, D, true);
      ep.col_bias = h->post_proj.bias;
      ep.row_zero = hm ? plan->mask_dev : nullptr;
      if (!b.linear("post_extract_proj", fln.op, N, E, h->post_proj.w, ep)) return false;
    } else {
      float* gm = h->fuse_ln_g; float* be = h->fuse_ln_b;
      b.push("fuse_ln", [=](cudaStream_t s) {
        return launch_layernorm(fused, DT_F32, E, gm, be, 1e-5f, x0, nullptr, DT_BF16, hm ? pl->mask_dev : nullptr, N, E, s);
      });
    }
    if (p_in > 0.f)      // features = self.dropout_input(features), hubert.py:729
      b.push("dropout", [=](cudaStream_t s) { return launch_dropout_residual(nullptr, x0, x0, N * D, p_in, seed, 1u, s); });
  } else {
    b.push_direct("load_features", [=](cudaStream_t s) {
      return launch_load_rows(pl->args.xin, pl->args.xin_dt, x0, hm ? pl->mask_dev : nullptr, N, D, s);
    });
  }
  const int G = 64, Tp = T + G;
  const long long pad_rows = (long long)B * Tp;
  const int KT = c.conv_pos, win = h->pos_window;
  void* xpad = b.alloc((size_t)pad_rows * P * D * 2);         // zero-gapped operand layout of the positional conv
  {
    const int planes = P;
    b.push("pos_pad", [=](cudaStream_t s) { return launch_split_rows(x0, D, xpad, planes, N, D, T, Tp, s); });
    std::vector<Tap> taps;
    for (int k = 0; k < KT; ++k) taps.push_back(Tap{k - KT / 2, 0, k * win});
    Epilogue ep = epilogue(cpre, D, true);
    ep.col_bias = h->pos_bias;
    ep.map_mode = MAP_2LEVEL; ep.S2 = Tp; ep.S1 = Tp; ep.H = 1; ep.W = T; ep.O2 = T; ep.O1 = 0; ep.O0 = 0;
    if (!b.gemm("pos_conv", xpad, pad_rows, P * D, h->pos_w, pad_rows, taps, win / 64, D, ep, 64, h->pos_acol)) return false;
    float* x1 = xin[0];
    if (post) {          // x = F.dropout(LN(x + GELU(conv(x)))), wav2vec2.py:872-879
      float* gm = h->enc_ln_g; float* be = h->enc_ln_b;
      b.push("gelu", [=](cudaStream_t s) { return launch_gelu_fwd(cpre, DT_F32, x0, spre, DT_F32, N * D, s); });
      b.push("layer_ln", [=](cudaStream_t s) {
        return launch_layernorm(spre, DT_F32, D, gm, be, 1e-5f, x1, nullptr, DT_BF16, nullptr, N, D, s);
      });
      if (p_enc > 0.f)
        b.push("dropout", [=](cudaStream_t s) { return launch_dropout_residual(nullptr, x1, x1, N * D, p_enc, seed, 2u, s); });
    } else if (p_enc > 0.f)     // x = F.dropout(x + GELU(conv(x))), wav2vec2.py:879
      b.push("gelu", [=](cudaStream_t s) { return launch_masked_gelu(cpre, DT_F32, x0, x1, DT_F32, N * D, p_enc, seed, 2u, s); });
    else
      b.push("gelu", [=](cudaStream_t s) { return launch_gelu_fwd(cpre, DT_F32, x0, x1, DT_F32, N * D, s); });
  }
  for (int l = 0; l < L; ++l) {
    const LayerW& lw = h->layers[l];
    b.cur_layer = l;
    float* x = xin[l];
    if (ldrop) {
      float* xn = xin[l + 1];
      b.push_on_drop("layerdrop", [=](cudaStream_t s) {
        return cudaMemcpyAsync(xn, x, (size_t)N * D * 4, cudaMemcpyDeviceToDevice, s) == cudaSuccess ? 0 : 1;
      });
    }
    const unsigned site = 16u + 4u * (unsigned)l;
    // block output + bias into dtmp, then target = res + m * dtmp (dropout1 / dropout3, wav2vec2.py:980,990)
    auto block_dropout = [&](const float* res, float* target, unsigned st) {
      b.push("dropout", [=](cudaStream_t s) { return launch_dropout_residual(res, dtmp, target, N * D, p_enc, seed, st, s); });
    };
    // post-LN: the qkv GEMM reads x_l itself; its operand form is made here, in layer l's own steps, so that a
    // dropped layer's on-drop copy is all LayerDrop needs
    if (post) b.split(x, D, h1[l].op, N, D);
    else b.layernorm("layer_ln", x, DT_F32, lw.ln1_g, lw.ln1_b, 1e-5f, h1[l]);
    {
      Epilogue ep = epilogue(qkv[l].data, 3 * D, f32);
      ep.col_bias = lw.qkv.bias;
      if (!b.linear("qkv_proj", h1[l].op, N, D, lw.qkv.w, ep)) return false;
      const char* q = reinterpret_cast<const char*>(qkv[l].data);
      void* o = ctx[l].data;
      float* ls = lse[l];
      b.push("attention", [=](cudaStream_t s) {
        if (!f32)      // bf16 mode: the mma.sync forward kernel, also writing the log-sum-exp of every query row
          return launch_attention(q, hm ? pl->mask_dev : nullptr, o, B, T, D, Hh, 0, s, ls);
        return launch_attention_x(q, 3 * D, q + (size_t)D * es, 3 * D, q + (size_t)2 * D * es, 3 * D, act_dt,
                                  hm ? pl->mask_dev : nullptr, o, D, act_dt, B, Hh, T, T, 1.0f, s, ls);
      });
      b.sync_op(ctx[l]);
    }
    if (p_enc > 0.f) {
      Epilogue ep = epilogue(dtmp, D, true);
      ep.col_bias = lw.out.bias;
      if (!b.linear("out_proj", ctx[l].op, N, D, lw.out.w, ep)) return false;
      block_dropout(x, xmid[l], site);
    } else {
      Epilogue ep = epilogue(xmid[l], D, true);
      ep.col_bias = lw.out.bias; ep.R = x; ep.ldr = D; ep.r_fp32 = 1;
      if (!b.linear("out_proj", ctx[l].op, N, D, lw.out.w, ep)) return false;
    }
    if (post) {          // y1 = self_attn_layer_norm(r1): fp32 residual stream of the FFN block + the fc1 operand
      const float* r1 = xmid[l]; float* yv = y1[l];
      void* yl = f32 ? nullptr : h2[l].data;
      const float* gm = lw.ln1_g; const float* be = lw.ln1_b;
      b.push("layer_ln", [=](cudaStream_t s) {
        return launch_layernorm(r1, DT_F32, D, gm, be, 1e-5f, yv, yl, DT_BF16, nullptr, N, D, s);
      });
      b.sync_op(h2[l]);
    } else {
      b.layernorm("layer_ln", xmid[l], DT_F32, lw.ln2_g, lw.ln2_b, 1e-5f, h2[l]);
    }
    {
      Epilogue ep = epilogue(u[l].data, F, f32);
      ep.col_bias = lw.fc1.bias;
      if (!b.linear("fc1", h2[l].op, N, D, lw.fc1.w, ep)) return false;
      const void* uu = u[l].data; void* gg = g[l].data;
      if (p_act > 0.f)   // dropout2 = activation_dropout after the GELU, wav2vec2.py:987
        b.push("gelu", [=](cudaStream_t s) {
          return launch_masked_gelu(uu, act_dt, nullptr, gg, act_dt, N * F, p_act, seed, site + 1u, s);
        });
      else
        b.push("gelu", [=](cudaStream_t s) { return launch_gelu_fwd(uu, act_dt, nullptr, gg, act_dt, N * F, s); });
      b.sync_op(g[l]);
    }
    float* res2 = post ? y1[l] : xmid[l];          // FFN block: residual input, sum (post-LN: r2, before LN2)
    float* out2 = post ? r2[l] : xin[l + 1];
    if (p_enc > 0.f) {
      Epilogue ep = epilogue(dtmp, D, true);
      ep.col_bias = lw.fc2.bias;
      if (!b.linear("fc2", g[l].op, N, F, lw.fc2.w, ep)) return false;
      block_dropout(res2, out2, site + 2u);
    } else {
      Epilogue ep = epilogue(out2, D, true);
      ep.col_bias = lw.fc2.bias; ep.R = res2; ep.ldr = D; ep.r_fp32 = 1;
      if (!b.linear("fc2", g[l].op, N, F, lw.fc2.w, ep)) return false;
    }
    if (post) {          // x_{l+1} = final_layer_norm(r2)
      float* xn = xin[l + 1];
      const float* gm = lw.ln2_g; const float* be = lw.ln2_b;
      b.push("layer_ln", [=](cudaStream_t s) {
        return launch_layernorm(out2, DT_F32, D, gm, be, 1e-5f, xn, nullptr, DT_BF16, nullptr, N, D, s);
      });
    }
  }
  b.cur_layer = -1;
  {
    float* xl = xin[L];
    float* gm = h->enc_ln_g; float* be = h->enc_ln_b;
    if (post)            // no final LayerNorm after post-LN layers (wav2vec2.py:862-863)
      b.push_direct("output", [=](cudaStream_t s) { return launch_convert(xl, DT_F32, pl->args.out, pl->args.out_dt, N * D, s); });
    else
      b.push_direct("final_ln", [=](cudaStream_t s) {
        return launch_layernorm(xl, DT_F32, D, gm, be, 1e-5f, nullptr, pl->args.out, pl->args.out_dt, nullptr, N, D, s);
      });
  }
  if (!sizing) plan->fwd_steps = plan->steps.size();

  // ================================================================ backward
  float2* stats = reinterpret_cast<float2*>(b.alloc((size_t)N * 8));
  float* Dbuf = b.f32buf((long long)B * Hh * T);
  float* dx = post ? dy : b.f32buf(N * D);  // gradient of the residual stream (ping; post-LN: starts as dL/dy itself)
  float* dxm = b.f32buf(N * D);            // ... at the middle of a layer (pong)
  float* dh = b.f32buf(N * D);             // gradient of a LayerNorm output
  Act dxa = b.act(N, D);                   // operand form of dx / dxm
  Act dga = b.act(N, F);                   // dL/dg
  Act dua = b.act(N, F);                   // dL/du
  Act dctx = b.act(N, D);
  Act dqkv = b.act(N, 3 * D);
  void* tA = b.alloc((size_t)std::max(3 * D, F) * P * Kp * 2);      // transposed dY operand
  void* tB = b.alloc((size_t)std::max(std::max(D, F), E) * P * Kp * 2);      // transposed X operand
  // dX [N, n_in] = dY [N, n_out] W: A = dY operand, B = W^T (packed [n_in, n_out])
  auto dgrad = [&](const void* dy_op, int n_out, const LinearW& wT, void* out, bool out_f32, const char* tag) {
    return b.linear(tag, dy_op, N, n_out, wT.w, epilogue(out, wT.w.n, out_f32));
  };
  // dW [n_out, n_in] = dY^T X (+ bias gradient = column sums of dY)
  auto wgrad = [&](const void* dyv, int dy_dt, int n_out, const void* xv, int x_dt, int n_in, float* dW, float* db, const char* tag) {
    const int planes = P;
    b.push("transpose", [=](cudaStream_t s) { return launch_transpose_split(dyv, dy_dt, n_out, N, n_out, tA, planes, Kp, 1.0f, s); });
    b.push("transpose", [=](cudaStream_t s) { return launch_transpose_split(xv, x_dt, n_in, N, n_in, tB, planes, Kp, 1.0f, s); });
    PackedW xw;
    xw.w = reinterpret_cast<bf16*>(tB); xw.n = n_in; xw.k = (int)Kp; xw.kpad = (int)Kp;
    // whole tiles, no stream-K: measured faster for the encoder's weight gradients (64-256 tiles of 19 K blocks at
    // 8 x 150 tokens), 15.96 vs 16.96 ms per frozen-extractor step (73 launches at ~13 us against 24.5 us with
    // stream-K: the partial-tile round trip through the workspace costs more than the idle SMs)
    if (!b.linear(tag, tA, n_out, (int)Kp, xw, epilogue(dW, n_in, true))) return false;
    if (db != nullptr)
      b.push("bias_grad", [=](cudaStream_t s) { return launch_colsum(dyv, dy_dt, n_out, N, n_out, db, 1.0f, s); });
    return true;
  };
  const float qscale = 1.0f / std::sqrt(64.0f);
  const long long LG = enc_layer_grad_floats(D, F);
  // (the caller's dL/dy is staged into `dy` by avh_encoder_backward before the steps run)
  if (!post) {   // final LayerNorm
    float* gfin = grads + (long long)L * LG;
    float* xl = xin[L];
    float* gm = h->enc_ln_g;
    b.push("ln_bwd", [=](cudaStream_t s) { return launch_ln_bwd(xl, gm, dy, nullptr, dx, stats, gfin, gfin + D, N, D, 1e-5f, s); });
  }
  for (int l = L - 1; l >= 0; --l) {
    const LayerW& lw = h->layers[l];
    b.cur_layer = l;
    float* gl = grads + (long long)l * LG;
    float* g_qkv_w = gl;                         // [3D, D]
    float* g_qkv_b = g_qkv_w + 3ll * D * D;      // [3D]
    float* g_out_w = g_qkv_b + 3ll * D;          // [D, D]
    float* g_out_b = g_out_w + (long long)D * D;
    float* g_ln1 = g_out_b + D;                  // gamma, beta
    float* g_fc1_w = g_ln1 + 2ll * D;            // [F, D]
    float* g_fc1_b = g_fc1_w + (long long)F * D;
    float* g_fc2_w = g_fc1_b + F;                // [D, F]
    float* g_fc2_b = g_fc2_w + (long long)D * F;
    float* g_ln2 = g_fc2_b + D;
    const unsigned site = 16u + 4u * (unsigned)l;
    if (ldrop)      // a dropped layer passes dx through unchanged; its parameters get zero gradients
      b.push_on_drop("layerdrop", [=](cudaStream_t s) {
        return cudaMemsetAsync(gl, 0, (size_t)LG * 4, s) == cudaSuccess ? 0 : 1;
      });
    // gradient of a block output behind a dropout: dtmp = m * dy and its operand form, or (p = 0) dy and its split
    auto block_grad = [&](float* dyv, unsigned st) -> float* {
      if (p_enc <= 0.f) {
        b.split(dyv, D, dxa.op, N, D);
        return dyv;
      }
      void* op = dxa.op;
      const int planes = P;
      b.push("dropout_bwd", [=](cudaStream_t s) { return launch_dropout_grad(dyv, dtmp, op, planes, N, D, p_enc, seed, st, s); });
      return dtmp;
    };
    // post-LN: gradient of a LayerNorm input r = res + m * block from its output's gradients (dya + dyb), written to
    // dr, with m * dr into dtmp (p > 0) and its operand form; returns what the block's weight gradient reads
    auto post_ln_grad = [&](const float* r, const float* gm, const float* dya, const float* dyb, float* dr, float* g_ln,
                            unsigned st) -> float* {
      float* mo = p_enc > 0.f ? dtmp : nullptr;
      void* op = dxa.op;
      const int planes = P;
      b.push("ln_bwd", [=](cudaStream_t s) {
        return launch_ln_post_bwd(r, gm, dya, dyb, dr, mo, op, planes, stats, g_ln, g_ln + D, N, D, 1e-5f, p_enc, seed, st, s);
      });
      return mo ? mo : dr;
    };
    // ---- fc2: x' = xm + m (g W2^T + b2)   (post-LN: r2 = y1 + m (g W2^T + b2), x' = LN2(r2); dr2 -> dxm)
    if (post) {
      float* d3 = post_ln_grad(r2[l], lw.ln2_g, dx, nullptr, dxm, g_ln2, site + 2u);
      if (!wgrad(d3, DT_F32, D, g[l].data, act_dt, F, g_fc2_w, g_fc2_b, "fc2_wgrad")) return false;
    } else if (p_enc > 0.f) {
      float* d3 = block_grad(dx, site + 2u);
      if (!wgrad(d3, DT_F32, D, g[l].data, act_dt, F, g_fc2_w, g_fc2_b, "fc2_wgrad")) return false;
    } else {
      if (!wgrad(dx, DT_F32, D, g[l].data, act_dt, F, g_fc2_w, g_fc2_b, "fc2_wgrad")) return false;
      block_grad(dx, site + 2u);
    }
    if (!dgrad(dxa.op, D, lw.fc2T, dga.data, f32, "fc2_dgrad")) return false;
    {
      const void* uu = u[l].data; const void* dgv = dga.data; void* duv = dua.data;
      if (p_act > 0.f)
        b.push("gelu_bwd", [=](cudaStream_t s) {
          return launch_masked_gelu_bwd(uu, act_dt, dgv, act_dt, duv, act_dt, N * F, p_act, seed, site + 1u, s);
        });
      else
        b.push("gelu_bwd", [=](cudaStream_t s) { return launch_gelu_bwd(uu, act_dt, dgv, act_dt, duv, act_dt, N * F, s); });
      b.sync_op(dua);
    }
    // ---- fc1: u = h2 W1^T + b1
    if (!wgrad(dua.data, act_dt, F, h2[l].data, act_dt, D, g_fc1_w, g_fc1_b, "fc1_wgrad")) return false;
    if (!dgrad(dua.op, F, lw.fc1T, dh, true, "fc1_dgrad")) return false;
    // ---- out_proj: xm = x + m (ctx Wo^T + bo)   (post-LN: r1 = x + m (ctx Wo^T + bo), y1 = LN1(r1); dr1 -> dx)
    if (post) {
      float* d1 = post_ln_grad(xmid[l], lw.ln1_g, dxm, dh, dx, g_ln1, site);
      if (!wgrad(d1, DT_F32, D, ctx[l].data, act_dt, D, g_out_w, g_out_b, "out_wgrad")) return false;
    } else {
      {   // LN2: dxm = dx + dLN(dh; xm)
        float* xm = xmid[l]; float* gm = lw.ln2_g;
        b.push("ln_bwd", [=](cudaStream_t s) { return launch_ln_bwd(xm, gm, dh, dx, dxm, stats, g_ln2, g_ln2 + D, N, D, 1e-5f, s); });
      }
      if (p_enc > 0.f) {
        float* d1 = block_grad(dxm, site);
        if (!wgrad(d1, DT_F32, D, ctx[l].data, act_dt, D, g_out_w, g_out_b, "out_wgrad")) return false;
      } else {
        if (!wgrad(dxm, DT_F32, D, ctx[l].data, act_dt, D, g_out_w, g_out_b, "out_wgrad")) return false;
        block_grad(dxm, site);
      }
    }
    if (!dgrad(dxa.op, D, lw.outT, dctx.data, f32, "out_dgrad")) return false;
    {   // attention
      const char* q = reinterpret_cast<const char*>(qkv[l].data);
      char* dq = reinterpret_cast<char*>(dqkv.data);
      const void* dO = dctx.data; const void* O = ctx[l].data;
      float* ls = lse[l];
      b.push("attention_bwd", [=](cudaStream_t s) {
        if (!f32)      // bf16 mode: tensor-core backward (attention.cu); fp32 mode: the fp32 CUDA-core kernels
          return launch_attention_bwd_tc(q, dO, O, ls, hm ? pl->mask_dev : nullptr, dq, Dbuf, B, T, D, Hh, s);
        return launch_attention_bwd(q, 3 * D, q + (size_t)D * es, 3 * D, q + (size_t)2 * D * es, 3 * D, act_dt, dO, O, D, act_dt, ls,
                                    hm ? pl->mask_dev : nullptr, dq, dq + (size_t)D * es, dq + (size_t)2 * D * es, 3 * D, act_dt,
                                    Dbuf, B, Hh, T, s);
      });
      b.sync_op(dqkv);
    }
    // ---- qkv: [q', k, v] = h1 Wqkv'^T + b' with q' = s q (the scaling is folded into Wq', bq')
    if (!wgrad(dqkv.data, act_dt, 3 * D, h1[l].data, act_dt, D, g_qkv_w, g_qkv_b, "qkv_wgrad")) return false;
    b.push("scale", [=](cudaStream_t s) {     // d/dWq = s d/dWq', d/dbq = s d/dbq'
      if (launch_scale(g_qkv_w, (long long)D * D, qscale, s)) return 1;
      return launch_scale(g_qkv_b, D, qscale, s);
    });
    if (post) {          // dx_l = dr1 + dL/dx_l through the qkv projection: the dgrad accumulates onto dx
      Epilogue ep = epilogue(dx, D, true);
      ep.R = dx; ep.ldr = D; ep.r_fp32 = 1;
      if (!b.linear("qkv_dgrad", dqkv.op, N, 3 * D, lw.qkvT.w, ep)) return false;
    } else {
      if (!dgrad(dqkv.op, 3 * D, lw.qkvT, dh, true, "qkv_dgrad")) return false;
      {   // LN1: dx = dxm + dLN(dh; x)
        float* xl = xin[l]; float* gm = lw.ln1_g;
        b.push("ln_bwd", [=](cudaStream_t s) { return launch_ln_bwd(xl, gm, dh, dxm, dx, stats, g_ln1, g_ln1 + D, N, D, 1e-5f, s); });
      }
    }
    if (l % 4 == 0) {      // layers l .. l+3 are final: one gradient bucket (Large: 4 x 12.6 M floats)
      b.cur_layer = -1;
      grad_mark((long long)l * LG, (long long)std::min(L, l + 4) * LG);
    }
  }
  b.cur_layer = -1;
  // ---- positional conv block: x1 = m2 (x0 + GELU(c)), c = conv(x0) + bias  (pos-conv weight gradients: see posconv_bwd)
  //      post-LN: x1 = m2 LN(s), s = x0 + GELU(c)
  {
    float* gpos = grads + (long long)L * LG + 2ll * D;       // bias [D], weight_g [KT], weight_v [D, D/G, KT]
    if (p_enc > 0.f)     // dx = m2 dL/dx1 in place: the gradient of both the residual and the GELU input
      b.push("dropout_bwd", [=](cudaStream_t s) { return launch_dropout_grad(dx, dx, nullptr, 1, N, D, p_enc, seed, 2u, s); });
    float* ds = dx;                                          // dL/d(x0 + GELU(c))
    if (post) {          // encoder.layer_norm: ds = LN^T(m2 dL/dx1; s) into dxm, its gamma / beta into their usual slot
      float* gfin = grads + (long long)L * LG;
      float* gm = h->enc_ln_g;
      b.push("ln_bwd", [=](cudaStream_t s) { return launch_ln_bwd(spre, gm, dx, nullptr, dxm, stats, gfin, gfin + D, N, D, 1e-5f, s); });
      ds = dxm;
    }
    float* dc = dh;                                          // dL/dc = ds * GELU'(c)
    b.push("gelu_bwd", [=](cudaStream_t s) { return launch_gelu_bwd(cpre, DT_F32, ds, DT_F32, dc, DT_F32, N * D, s); });
    b.push("bias_grad", [=](cudaStream_t s) { return launch_colsum(dc, DT_F32, D, N, D, gpos, 1.0f, s); });
    // dgrad: dx0[t, i] = dx[t, i] + sum_k sum_o dc[t + 64 - k, o] w[o, i, k]: the same shifted-row GEMM over the
    // zero-gapped layout with the taps mirrored and the weights transposed inside every group (pos_wT)
    void* dcpad = b.alloc((size_t)pad_rows * P * D * 2);     // zero-gapped operand layout of dL/dc (gap rows stay zero)
    const int planes = P;
    b.push("pos_pad", [=](cudaStream_t s) { return launch_split_rows(dc, D, dcpad, planes, N, D, T, Tp, s); });
    std::vector<Tap> taps;
    for (int k = 0; k < KT; ++k) taps.push_back(Tap{KT / 2 - k, 0, k * win});
    Epilogue ep = epilogue(dxo, D, true);
    ep.R = ds; ep.ldr = D; ep.r_fp32 = 1;
    ep.row_zero = hm ? plan->mask_dev : nullptr;             // x0 = index_put(features, mask, 0): no gradient into pad rows
    ep.map_mode = MAP_2LEVEL; ep.S2 = Tp; ep.S1 = Tp; ep.H = 1; ep.W = T; ep.O2 = T; ep.O1 = 0; ep.O0 = 0;
    if (!b.gemm("pos_conv_dgrad", dcpad, pad_rows, P * D, h->pos_wT, pad_rows, taps, win / 64, D, ep, 64, h->pos_acol)) return false;
    // weight gradients of the grouped convolution + weight-norm backward
    if (!posconv_wgrad(b, h, dc, x0, N, B, T, gpos + D, gpos + D + KT)) return false;
    if (tail) {
      // dxo = dL/dx0 (rows of padded frames already zero).  post_extract_proj: x0 = m1 (fln Wp^T + bp); then the fusion
      // LayerNorm (its input comes from the frozen extractors: only dgamma / dbeta are needed)
      float* gt = gpos + D + KT + (long long)D * (D / c.conv_pos_groups) * KT;
      float* dfl = nullptr;
      float* g_ln = gt;
      const bool pp = h->has_post_proj;
      if (p_in > 0.f) {  // dxo = m1 dxo in place (+ the operand form post_extract_proj's dgrad reads)
        void* op = pp ? dxa.op : nullptr;
        const int planes = P;
        b.push("dropout_bwd", [=](cudaStream_t s) { return launch_dropout_grad(dxo, dxo, op, planes, N, D, p_in, seed, 1u, s); });
      }
      if (pp) {
        float* g_pw = gt; float* g_pb = gt + (long long)D * E;
        g_ln = g_pb + D;
        if (!wgrad(dxo, DT_F32, D, fln.data, act_dt, E, g_pw, g_pb, "post_proj_wgrad")) return false;
        if (p_in <= 0.f) b.split(dxo, D, dxa.op, N, D);
        dfl = b.f32buf(N * E);
        if (!dgrad(dxa.op, D, h->post_projT, dfl, true, "post_proj_dgrad")) return false;
      } else {
        dfl = dxo;
      }
      float* dfused = b.f32buf(N * E);       // dL/d(fused): used by mode 2, a by-product otherwise
      float* gm = h->fuse_ln_g;
      b.push("ln_bwd", [=](cudaStream_t s) { return launch_ln_bwd(fused, gm, dfl, nullptr, dfused, stats, g_ln, g_ln + E, N, E, 1e-5f, s); });
      // final LayerNorm, positional conv, post_extract_proj, fusion LayerNorm: one bucket; the feature extractors' another
      grad_mark((long long)L * LG, full ? (g_ln + 2ll * E) - grads : GF);
      if (full) {
        // ============================================================ backward of the feature extractors (mode 2)
        float* gf = g_ln + 2ll * E;                         // frontend gradients follow layer_norm.{weight,bias}
        if (key.pen) {      // features_pen = fused.pow(2).mean() (hubert.py:629) enters the extractors through GradMultiply too
          float* dp = b.f32buf(4);
          if (!sizing) plan->dpen = dp;
          const float* fu = fused;
          const float sc = 2.0f / (float)(N * E);
          b.push("pen_grad", [=](cudaStream_t s) { return launch_pen_grad(fu, dfused, N * E, dp, sc, s); });
        }
        b.push("scale", [=](cudaStream_t s) {               // GradMultiply on the extractor outputs (grad_multiply.py:105-114)
          return pl->fgm != 1.f ? launch_scale(dfused, N * E, pl->fgm, s) : 0;
        });
        // generic dW [n_out, n_in] (+)= dY^T X over `rows` rows; X either a plain matrix (x_op = false) or an operand-form
        // matrix [rows, P * n_in] (planes side by side); K = rows is cut into segments the GEMM's K-step table holds
        long long max_a = (long long)D * ((N + 63) / 64 * 64), max_b = (long long)std::max(Fp, 512) * ((N + 63) / 64 * 64);
        if (key.has_video) {
          max_a = std::max(max_a, 64ll * ((nfr * 1936 + 63) / 64 * 64));
          max_b = std::max(max_b, 320ll * ((nfr * 1936 + 63) / 64 * 64));
          int cin = 64, Hh2 = 22;
          for (int L = 0; L < 4; ++L) {
            const int C = 64 << L;
            const int Ho = L == 0 ? 22 : (Hh2 + 2 - 3) / 2 + 1;
            const long long kp = (nfr * Ho * Ho + 63) / 64 * 64;
            max_a = std::max(max_a, (long long)C * kp);
            max_b = std::max(max_b, (long long)9 * std::max(cin, C) * kp);
            cin = C; Hh2 = Ho;
          }
        }
        void* ftA = b.alloc((size_t)max_a * P * 2);
        void* ftB = b.alloc((size_t)max_b * P * 2);
        // x_mode: 0 = xv [rows, n_in] values (x_dt), 1 = xv operand planes (bf16 [rows, P * n_in]), 2 = ftB already holds
        // the transposed operand (im2colT)
        auto wgrad_rows = [&](const void* dyv, long long ld_dy, int n_out, const void* xv, int x_dt, long long ld_x, int x_mode,
                              int n_in, long long rows, float* dW, float* db, const char* tag, int dy_dt = DT_F32) -> bool {
          const long long kp = (rows + 63) / 64 * 64;
          const int planes = P;
          if (!f32 && n_out % 8 == 0 && ld_dy % 8 == 0) {
            b.push("transpose", [=](cudaStream_t s) { return launch_transposeT(dyv, dy_dt, ld_dy, rows, n_out, ftA, kp, kp, s); });
          } else {
            b.push("transpose", [=](cudaStream_t s) {
              return launch_transpose_split(dyv, dy_dt, ld_dy, rows, n_out, ftA, planes, kp, 1.0f, s);
            });
          }
          if (x_mode == 1) {
            for (int pp = 0; pp < P; ++pp) {
              const __nv_bfloat16* src = reinterpret_cast<const __nv_bfloat16*>(xv) + (long long)pp * n_in;
              __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(ftB) + (long long)pp * kp;
              if (!f32 && n_in % 8 == 0 && ld_x % 8 == 0)
                b.push("transpose", [=](cudaStream_t s) { return launch_transposeT(src, DT_BF16, ld_x, rows, n_in, dst, kp, kp, s); });
              else
                b.push("transpose", [=](cudaStream_t s) {
                  return launch_transpose_split(src, DT_BF16, ld_x, rows, n_in, dst, 1, kp, 1.0f, s, 0, 0, (long long)planes * kp);
                });
            }
          } else if (x_mode == 0) {
            if (!f32 && x_dt == DT_BF16 && n_in % 8 == 0 && ld_x % 8 == 0)
              b.push("transpose", [=](cudaStream_t s) { return launch_transposeT(xv, DT_BF16, ld_x, rows, n_in, ftB, kp, kp, s); });
            else
              b.push("transpose", [=](cudaStream_t s) {
                return launch_transpose_split(xv, x_dt, ld_x, rows, n_in, ftB, planes, kp, 1.0f, s);
              });
          }
          if (!f32) {
            // bf16 mode: ONE launch over the whole K extent (no step table), stream-K over the SMs: the output is a handful
            // of tiles (dW of a 64-channel conv: 1 x 5) while K is the pixel count (580 800 in layer1 at 8 x 150 frames)
            PackedW xw;
            xw.w = reinterpret_cast<bf16*>(ftB); xw.n = n_in; xw.k = (int)kp; xw.kpad = (int)kp;
            b.linear_k = true; b.force_sk = 1;
            const bool ok = b.gemm(tag, ftA, n_out, (int)kp, xw, n_out, {Tap{0, 0, 0}}, (int)(kp / 64), (int)kp,
                                   epilogue(dW, n_in, true), 0, nullptr, kp);
            b.linear_k = false; b.force_sk = 0;
            if (!ok) return false;
          } else {
            const long long seg = 256 * 64;
            for (long long k0 = 0; k0 < kp; k0 += seg) {
              const long long kl = std::min(seg, kp - k0);
              PackedW xw;
              xw.w = reinterpret_cast<bf16*>(ftB) + k0; xw.n = n_in; xw.k = (int)kp; xw.kpad = (int)kp;
              Epilogue ep = epilogue(dW, n_in, true);
              if (k0 > 0) { ep.R = dW; ep.ldr = n_in; ep.r_fp32 = 1; }
              const char* a = reinterpret_cast<const char*>(ftA) + (size_t)k0 * 2;
              if (!b.gemm(tag, a, n_out, (int)(P * kp - k0), xw, n_out, {Tap{0, 0, 0}}, (int)(kl / 64), (int)kp, ep, 0, nullptr, P * kp))
                return false;
            }
          }
          if (db != nullptr)
            b.push("bias_grad", [=](cudaStream_t s) { return launch_colsum(dyv, dy_dt, ld_dy, rows, n_out, db, 1.0f, s); });
          return true;
        };
        // a dropped modality arm (0 * features): its backward is skipped, its gradients are zeros
        auto zero_grads_on_drop = [&](int mod, float* begin, float* end) {
          b.cur_mod = mod;
          b.push_on_drop("modality_drop", [=](cudaStream_t s) {
            return cudaMemsetAsync(begin, 0, (size_t)(end - begin) * 4, s) == cudaSuccess ? 0 : 1;
          });
          b.cur_mod = 0;
        };
        if (key.has_audio) {
          float* g_w = gf; float* g_b = g_w + (long long)D * Fp;
          gf = g_b + D;
          if (key.moddrop) b.cur_mod = 1;
          if (!wgrad_rows(dfused, E, D, arows.data, act_dt, Fp, 0, Fp, N, g_w, g_b, "proj_audio_wgrad")) return false;
          b.cur_mod = 0;
          if (key.moddrop) zero_grads_on_drop(1, g_w, gf);
        }
        if (key.has_video) {
          float* g_video = gf;
          if (key.moddrop) b.cur_mod = 2;
          float* g_w = gf; float* g_b = g_w + (long long)D * 512;
          gf = g_b + D;
          if (!wgrad_rows(dfused + v_off, E, D, feat.data, act_dt, 512, 0, 512, N, g_w, g_b, "proj_video_wgrad")) return false;
          // d(feat) = d(fused_video) Wv
          b.split(dfused + v_off, E, dxa.op, N, D);
          float* dfeat = b.f32buf(N * 512);
          if (!dgrad(dxa.op, D, h->proj_vT, dfeat, true, "proj_video_dgrad")) return false;
          // gradient slots of the ResNet, in forward (state-dict) order
          float* g_stem_w = gf; float* g_stem_bn = g_stem_w + 64 * 320; float* g_stem_slope = g_stem_bn + 128;
          gf = g_stem_slope + 64;
          struct BlockG { float *c1w, *bn1, *s1, *c2w, *bn2, *s2, *dsw, *dsbn; };
          BlockG bg[4][2];
          {
            int cin = 64;
            for (int L = 0; L < 4; ++L) {
              const int C = 64 << L;
              for (int bi = 0; bi < 2; ++bi) {
                BlockG& g = bg[L][bi];
                g.c1w = gf; gf += (long long)C * 9 * cin;
                g.bn1 = gf; gf += 2 * C;
                g.s1 = gf; gf += C;
                g.c2w = gf; gf += (long long)C * 9 * C;
                g.bn2 = gf; gf += 2 * C;
                g.s2 = gf; gf += C;
                g.dsw = nullptr; g.dsbn = nullptr;
                if (L > 0 && bi == 0) { g.dsw = gf; gf += (long long)C * cin; g.dsbn = gf; gf += 2 * C; }
                cin = C;
              }
            }
          }
          float* tot = b.f32buf(3 * 512);
          size_t dcol_elems = 0, dop_elems = 0;
          for (const ConvSave& cs : convs) {
            if (cs.cu == &h->stem) continue;
            const long long rows = nfr * cs.Ho * cs.Ho;
            dcol_elems = std::max(dcol_elems, (size_t)rows * cs.cu->ks * cs.cu->ks * cs.cu->cin);
            dop_elems = std::max(dop_elems, (size_t)rows * cs.cu->cout);
          }
          float* dcol = b.f32buf((long long)dcol_elems);
          void* dop = b.alloc(dop_elems * P * 2);
          // BatchNorm (+ residual) (+ PReLU) backward of one saved conv: dz -> d_raw (returned), d_res, parameter gradients
          const int graw_dt = f32 ? DT_F32 : DT_BF16;     // bf16 mode: d(raw conv output) is only ever a GEMM operand
          auto bn_bwd = [&](const ConvSave& cs, const float* dz, float* d_res, int res_acc, float* g_bn, float* g_slope) {
            const long long rows = nfr * cs.Ho * cs.Ho;
            const int Cc = cs.cu->cout;
            float* d_raw = b.f32buf(f32 ? rows * Cc : (rows * Cc + 1) / 2);
            const void* rawp = cs.raw.data;
            const void* resp = cs.res.data;
            const float* st = cs.stat; const float* gm = cs.cu->gamma; const float* bt = cs.cu->beta; const float* sl = cs.slope;
            b.push("bn_bwd", [=](cudaStream_t s) {
              return launch_bn_act_bwd(rawp, act_dt, resp, dz, st, gm, bt, sl, rows, Cc, bn_sums, tot, d_raw, d_res, res_acc,
                                       g_bn, g_bn + Cc, g_slope, s, graw_dt);
            });
            return d_raw;
          };
          // conv backward: dW = d_raw^T col(x); dx (+)= col2im(d_raw W)
          // d_raw: fp32 [rows, cout] in fp32 mode, bf16 in bf16 mode (graw_dt)
          auto conv_bwd = [&](const ConvSave& cs, const float* d_raw, float* dW, float* dx, int dx_acc) -> bool {
            const ConvUnit& cu = *cs.cu;
            const int K = cu.ks * cu.ks * cu.cin, Cc = cu.cout;
            const long long rows = nfr * cs.Ho * cs.Ho;
            const void* xin = cs.in.data;
            const int planes = P, ks = cu.ks, st = cu.stride, cin = cu.cin, H = cs.H, Ho = cs.Ho, pad = cs.pad;
            if (!f32) {
              // bf16 mode: the patches are written transposed straight from the map (no patch matrix, no transpose pass)
              const long long kp = (rows + 63) / 64 * 64;
              b.push("im2col", [=](cudaStream_t s) { return launch_im2colT(xin, nfr, H, cin, ks, st, pad, Ho, ftB, kp, s); });
              if (!wgrad_rows(d_raw, Cc, Cc, nullptr, DT_BF16, 0, 2, K, rows, dW, nullptr, "conv_wgrad", graw_dt)) return false;
            } else {
              b.push("im2col", [=](cudaStream_t s) {
                return launch_im2col2d(xin, act_dt, nfr, H, cin, ks, st, pad, Ho, colbuf, planes, s);
              });
              if (!wgrad_rows(d_raw, Cc, Cc, colbuf, DT_BF16, (long long)P * K, 1, K, rows, dW, nullptr, "conv_wgrad")) return false;
            }
            if (dx == nullptr) return true;
            const void* dopv = dop;
            if (f32) b.split(d_raw, Cc, dop, rows, Cc);
            else dopv = d_raw;                                     // already the bf16 operand
            // bf16 mode: patch gradients in bf16 (half the traffic)
            if (!b.linear("conv_dgrad", dopv, rows, Cc, cu.wT, epilogue(dcol, K, f32))) return false;
            b.push("col2im", [=](cudaStream_t s) { return launch_col2im2d(dcol, act_dt, nfr, H, cin, ks, st, pad, Ho, dx, dx_acc, s); });
            return true;
          };
          // avgpool
          float* dcur = b.f32buf(nfr * 9 * 512);
          {
            float* dc4 = dcur;
            b.push("avgpool_bwd", [=](cudaStream_t s) { return launch_avgpool_bwd(dfeat, dc4, nfr, 9, 512, s); });
          }
          // blocks in reverse; convs = [stem, (c1, [ds], c2) x 8]
          int ci = (int)convs.size() - 1;
          for (int L = 3; L >= 0; --L)
            for (int bi = 1; bi >= 0; --bi) {
              const BlockW& bw = h->blocks[L][bi];
              const BlockG& g = bg[L][bi];
              const ConvSave& c2 = convs[ci];
              const ConvSave* cd = bw.has_ds ? &convs[ci - 1] : nullptr;
              const ConvSave& c1 = convs[ci - (bw.has_ds ? 2 : 1)];
              ci -= bw.has_ds ? 3 : 2;
              const long long rows_out = nfr * c2.Ho * c2.Ho;
              const long long rows_in = nfr * c1.H * c1.H;
              float* d_res = b.f32buf(rows_out * c2.cu->cout);
              float* d_raw2 = bn_bwd(c2, dcur, d_res, 0, g.bn2, g.s2);
              float* d_a1 = b.f32buf(rows_out * c2.cu->cin);
              if (!conv_bwd(c2, d_raw2, g.c2w, d_a1, 0)) return false;
              float* d_raw1 = bn_bwd(c1, d_a1, nullptr, 0, g.bn1, g.s1);
              float* d_in = b.f32buf(rows_in * c1.cu->cin);
              if (L == 3 && bi == 1) {      // gradient maps of the last block, for the kink-attribution test
                b.stage("grad_layer4_1_conv2_in", d_a1, DT_F32, rows_out * 512);
                b.stage("grad_layer4_1_conv1_out", d_raw1, DT_F32, rows_out * 512);
              }
              if (!conv_bwd(c1, d_raw1, g.c1w, d_in, 0)) return false;
              if (cd != nullptr) {
                float* d_rawd = bn_bwd(*cd, d_res, nullptr, 0, g.dsbn, nullptr);
                if (!conv_bwd(*cd, d_rawd, g.dsw, d_in, 1)) return false;
              } else {
                const long long n_el = rows_in * c1.cu->cin;
                b.push("add", [=](cudaStream_t s) { return launch_add_f32(d_in, d_res, n_el, s); });
              }
              dcur = d_in;
            }
          // max-pool, stem BatchNorm + PReLU, stem weights
          {
            const ConvSave& cs = convs[0];
            float* d_act0 = b.f32buf(nfr * 1936 * 64);
            const void* a0 = act0.data;
            float* dp0 = dcur;
            b.push("maxpool_bwd", [=](cudaStream_t s) { return launch_maxpool_bwd(a0, act_dt, dp0, d_act0, nfr, 44, 64, 22, s, pool_arg); });
            float* d_raw0 = bn_bwd(cs, d_act0, nullptr, 0, g_stem_bn, g_stem_slope);
            if (!wgrad_rows(d_raw0, 64, 64, stemcol, DT_BF16, (long long)P * 320, 1, 320, nfr * 1936, g_stem_w, nullptr, "stem_wgrad",
                            graw_dt))
              return false;
          }
          b.cur_mod = 0;
          if (key.moddrop) zero_grads_on_drop(2, g_video, gf);
        }
        grad_mark((g_ln + 2ll * E) - grads, GF);         // modality projections + lip ResNet
      }
    } else {
      grad_mark((long long)L * LG, GF);                  // final LayerNorm + positional conv
    }
  }
  if (bytes_out) *bytes_out = b.sizer.used;
  return true;
}

// ============================================================================ Q-Former plan
// Qformer.bert(query_embeds, attention_mask, encoder_hidden_states, encoder_attention_mask) (src/model.py:611-617 ->
// src/sub_model/Qformer.py:805-968) for B clips x T query rows against Lk AV-feature rows each.  Post-LN BERT layers:
// x = LN(dense(SelfAttn(x)) + x); x = LN(dense(CrossAttn(x, enc)) + x); x = LN(fc2(GELU(fc1(x))) + x), eps 1e-12.
// Every Linear is a tcgen05 GEMM (the K / V projections of the AV features for ALL layers are one GEMM: they are
// ~80 % of the block's FLOPs); attention is launch_attention_x (qformer.cu).
bool build_qformer_plan(avh_handle* h, Plan* plan, bool sizing, size_t* bytes_out) {
  Builder b(h, plan, sizing);
  const avh_config& c = h->cfg;
  const PlanKey& key = plan->key;
  const bool f32 = b.f32;
  const int B = key.B, T = key.T, Lk = key.Lk, D = c.encoder_embed_dim, F = c.encoder_ffn_embed_dim;
  const int Hh = c.encoder_attention_heads, Ew = c.reserved[1], L = c.encoder_layers;
  const long long N = (long long)B * T, NK = (long long)B * Lk;
  const size_t es = b.es;
  const int act_dt = b.act_dt;
  const float eps = 1e-12f;                                   // BertConfig.layer_norm_eps
  Plan* pl = plan;
  unsigned char* qm = b.mask_buf(N);
  unsigned char* km = b.mask_buf(NK);
  if (!sizing) { plan->qmask_dev = qm; plan->kmask_dev = km; }
  float* x = b.f32buf(N * D);       // hidden states (fp32)
  float* tmp = b.f32buf(N * D);     // dense(...) + residual, before the LayerNorm
  float* emb = b.f32buf((long long)T * D);     // LayerNorm(query_tokens[:T])
  Act hbuf = b.act(N, D), qkv = b.act(N, 3 * D), cq = b.act(N, D), ctx = b.act(N, D), ffn = b.act(N, F);
  Act enc = b.act(NK, Ew), ckv = b.act(NK, 2 * D * L);
  const bool hm = key.has_mask;

  // ---- AV features -> operand form (the only step that reads a caller pointer besides the output store)
  {
    void* dst = enc.data;
    b.push_direct("load_features", [=](cudaStream_t s) { return launch_convert(pl->args.xin, pl->args.xin_dt, dst, act_dt, NK * Ew, s); });
  }
  b.sync_op(enc);
  // ---- embeddings: LayerNorm(query_embeds) (no position embeddings on the query-only path, Qformer.py:98-110)
  {
    const float* qt = h->qf_tokens; const float* g = h->qf_emb_g; const float* be = h->qf_emb_b;
    b.push("layer_ln", [=](cudaStream_t s) { return launch_layernorm(qt, DT_F32, D, g, be, eps, emb, nullptr, DT_BF16, nullptr, T, D, s); });
    b.push("layer_ln", [=](cudaStream_t s) { return launch_rows_broadcast(emb, x, (long long)T * D, B, s); });
  }
  // x = LayerNorm(tmp), then (unless it is the output) its operand copy
  auto post_ln = [&](const float* g, const float* be, bool to_op) {
    b.push("layer_ln", [=](cudaStream_t s) { return launch_layernorm(tmp, DT_F32, D, g, be, eps, x, nullptr, DT_BF16, nullptr, N, D, s); });
    if (to_op) b.split(x, D, hbuf.op, N, D);
  };
  auto dense_res = [&](const Act& a, int K, const LinearW& w, const char* tag) {      // tmp = a W^T + b + x
    Epilogue ep = epilogue(tmp, D, true);
    ep.col_bias = w.bias; ep.R = x; ep.ldr = D; ep.r_fp32 = 1;
    return b.linear(tag, a.op, N, K, w.w, ep);
  };
  b.split(x, D, hbuf.op, N, D);
  // ---- K / V of the AV features for every layer's cross-attention
  {
    Epilogue ep = epilogue(ckv.data, 2 * D * L, f32);
    ep.col_bias = h->qf_ckv.bias;
    if (!b.linear("cross_kv_proj", enc.op, NK, Ew, h->qf_ckv.w, ep)) return false;
  }
  const float scale = 0.125f;                                 // 1 / sqrt(attention_head_size = 64), Qformer.py:246
  for (int l = 0; l < L; ++l) {
    const QfLayerW& lw = h->qf_layers[l];
    b.cur_layer = l;
    {   // self-attention over the queries
      Epilogue ep = epilogue(qkv.data, 3 * D, f32);
      ep.col_bias = lw.sqkv.bias;
      if (!b.linear("qkv_proj", hbuf.op, N, D, lw.sqkv.w, ep)) return false;
      const char* q = reinterpret_cast<const char*>(qkv.data);
      void* o = ctx.data;
      b.push("attention", [=](cudaStream_t s) {
        return launch_attention_x(q, 3 * D, q + (size_t)D * es, 3 * D, q + (size_t)2 * D * es, 3 * D, act_dt, pl->qmask_dev, o, D,
                                  act_dt, B, Hh, T, T, scale, s);
      }, 4.0 * (double)B * Hh * (double)T * (double)T * 64.0);
      b.sync_op(ctx);
      if (!dense_res(ctx, D, lw.sout, "out_proj")) return false;
      post_ln(lw.ln1_g, lw.ln1_b, true);
    }
    {   // cross-attention to the AV features
      Epilogue ep = epilogue(cq.data, D, f32);
      ep.col_bias = lw.cq.bias;
      if (!b.linear("cross_q_proj", hbuf.op, N, D, lw.cq.w, ep)) return false;
      const void* q = cq.data;
      const char* kvp = reinterpret_cast<const char*>(ckv.data) + (size_t)l * 2 * D * es;
      const long long ldkv = 2ll * D * L;
      void* o = ctx.data;
      b.push("cross_attention", [=](cudaStream_t s) {
        return launch_attention_x(q, D, kvp, ldkv, kvp + (size_t)D * es, ldkv, act_dt, hm ? pl->kmask_dev : nullptr, o, D, act_dt,
                                  B, Hh, T, Lk, scale, s);
      }, 4.0 * (double)B * Hh * (double)T * (double)Lk * 64.0);
      b.sync_op(ctx);
      if (!dense_res(ctx, D, lw.cout, "cross_out_proj")) return false;
      post_ln(lw.ln2_g, lw.ln2_b, true);
    }
    {   // feed-forward of the query branch (intermediate_query / output_query, Qformer.py:482-485), erf GELU
      Epilogue ep = epilogue(ffn.data, F, f32);
      ep.col_bias = lw.fc1.bias; ep.act = ACT_GELU;
      if (!b.linear("fc1", hbuf.op, N, D, lw.fc1.w, ep)) return false;
      b.sync_op(ffn);
      if (!dense_res(ffn, F, lw.fc2, "fc2")) return false;
      post_ln(lw.ln3_g, lw.ln3_b, l + 1 < L);
    }
  }
  b.cur_layer = -1;
  b.push_direct("output", [=](cudaStream_t s) { return launch_convert(x, DT_F32, pl->args.out, pl->args.out_dt, N * D, s); });
  if (bytes_out) *bytes_out = b.sizer.used;
  return true;
}

constexpr int MAX_PLANS = 24;      // plans kept per handle (shape x stream); the least recently used one is evicted

void forget_plan(avh_handle* h, const Plan* p) {
  if (h->last_plan == p) h->last_plan = nullptr;
  if (h->prof_plan == p) h->prof_plan = nullptr;
}

Plan* get_plan(avh_handle* h, const PlanKey& key) {
  auto it = h->plans.find(key);
  if (it != h->plans.end()) {
    it->second->last_use = ++h->plan_clock;
    return it->second.get();
  }
  // bound workspace growth for ragged shape streams: evict the least recently used plan (one cudaFree, not all)
  while ((int)h->plans.size() >= MAX_PLANS) {
    auto victim = h->plans.begin();
    for (auto jt = h->plans.begin(); jt != h->plans.end(); ++jt)
      if (jt->second->last_use < victim->second->last_use) victim = jt;
    forget_plan(h, victim->second.get());
    h->plans.erase(victim);
  }
  if (key.training()) {
    // training plans keep every activation of the step (GBs for Large): at most two of them live per handle
    for (;;) {
      int n_train = 0;
      auto victim = h->plans.end();
      for (auto jt = h->plans.begin(); jt != h->plans.end(); ++jt)
        if (jt->first.training()) {
          ++n_train;
          if (victim == h->plans.end() || jt->second->last_use < victim->second->last_use) victim = jt;
        }
      if (n_train < 2) break;
      forget_plan(h, victim->second.get());
      h->plans.erase(victim);
    }
  }
  std::unique_ptr<Plan> p(new Plan());
  p->last_use = ++h->plan_clock;
  p->key = key;
  bool (*build)(avh_handle*, Plan*, bool, size_t*) = nullptr;
  switch (key.kind) {
    case PlanKind::Forward:
    case PlanKind::Ragged:
    case PlanKind::EncoderOnly:
    case PlanKind::TrainForward: build = build_plan; break;
    case PlanKind::EncoderTrain:
    case PlanKind::TailTrain:
    case PlanKind::FullTrain: build = build_encoder_train_plan; break;
    case PlanKind::QFormer: build = build_qformer_plan; break;
  }
  size_t bytes = 0;
  if (!build(h, p.get(), true, &bytes)) return nullptr;
  if (p->arena.init(bytes + (1 << 20))) return nullptr;
  if (!build(h, p.get(), false, nullptr)) return nullptr;
  if (key.kind == PlanKind::Ragged) {
    for (int i = 0; i < Plan::RAG_SLOTS; ++i) {
      if (cudaMallocHost(reinterpret_cast<void**>(&p->rag_host[i]), (size_t)p->rag_ints * 4) != cudaSuccess ||
          cudaEventCreateWithFlags(&p->rag_done[i], cudaEventDisableTiming) != cudaSuccess) {
        set_last_error("pinned descriptor allocation failed");
        return nullptr;
      }
    }
  }
  if (p->seed_dev != nullptr) {
    for (int i = 0; i < Plan::RAG_SLOTS; ++i) {
      if (cudaMallocHost(reinterpret_cast<void**>(&p->seed_host[i]), sizeof(unsigned long long)) != cudaSuccess ||
          cudaEventCreateWithFlags(&p->seed_done[i], cudaEventDisableTiming) != cudaSuccess) {
        set_last_error("pinned seed allocation failed");
        return nullptr;
      }
    }
  }
  Plan* raw = p.get();
  h->plans[key] = std::move(p);
  return raw;
}

int ensure_cap(void** p, size_t* cap, size_t bytes) {
  if (*cap >= bytes) return 0;
  if (*p) cudaFree(*p);
  *p = nullptr; *cap = 0;
  AVH_CUDA_OK(cudaMalloc(p, bytes));
  *cap = bytes;
  return 0;
}

bool ignorable_key(const std::string& k) {
  if (k == "mask_emb" || k == "label_embs_concat") return true;
  if (k.rfind("final_proj.", 0) == 0) return true;
  const std::string suf = "num_batches_tracked";
  return k.size() >= suf.size() && k.compare(k.size() - suf.size(), suf.size(), suf) == 0;
}
bool known_prefix(const std::string& k) {
  static const char* pre[] = {"feature_extractor_video.", "feature_extractor_audio.", "layer_norm.",
                              "post_extract_proj.", "encoder.", "embeddings.", "query_tokens"};
  for (const char* p : pre)
    if (k.rfind(p, 0) == 0) return true;
  return false;
}

}  // namespace
}  // namespace avh

// ============================================================================ extern "C"
extern "C" {

int avh_abi_version(void) { return AVH_ABI_VERSION; }
const char* avh_last_error(void) { return avh::g_err.c_str(); }
int64_t avh_launch_count(void) { return avh::g_launches.load(); }
void avh_reset_launch_count(void) { avh::g_launches.store(0); }
int64_t avh_graph_launch_count(void) { return avh::g_graph_launches.load(); }

int avh_create(const avh_config* cfg, int device, avh_handle** out) {
  AVH_CHECK(cfg != nullptr && out != nullptr, "null argument");
  AVH_CHECK(cfg->encoder_layers >= 1 && cfg->encoder_embed_dim >= 64, "bad encoder shape");
  AVH_CHECK(cfg->encoder_embed_dim % 64 == 0 && cfg->encoder_ffn_embed_dim % 64 == 0, "dims must be multiples of 64");
  AVH_CHECK(cfg->encoder_attention_heads * 64 == cfg->encoder_embed_dim, "head dim must be 64");
  AVH_CHECK(cfg->conv_pos >= 2 && cfg->conv_pos % 2 == 0 && cfg->conv_pos <= 128, "conv_pos must be even and <= 128");
  AVH_CHECK(cfg->conv_pos_groups >= 1 && cfg->encoder_embed_dim % cfg->conv_pos_groups == 0, "bad conv_pos_groups");
  AVH_CHECK(cfg->reserved[0] != 0 || (cfg->audio_feat_dim >= 1 && cfg->audio_feat_dim <= 1024), "bad audio_feat_dim");
  AVH_CHECK(cfg->modality_fuse == AVH_FUSE_CONCAT || cfg->modality_fuse == AVH_FUSE_ADD, "bad modality_fuse");
  AVH_CHECK(cfg->compute_mode == AVH_COMPUTE_BF16 || cfg->compute_mode == AVH_COMPUTE_FP32, "bad compute_mode");
  AVH_CHECK(cfg->reserved[0] >= 0 && cfg->reserved[0] <= 2, "reserved[0] must be 0 (AV-HuBERT), 1 (TransformerEncoder) or 2 (Q-Former)");
  AVH_CHECK(cfg->reserved[0] != 2 || (cfg->reserved[1] >= 64 && cfg->reserved[1] % 64 == 0 && cfg->reserved[2] >= 1),
            "Q-Former handles need reserved[1] = encoder_width (multiple of 64) and reserved[2] = query_tokens rows");
  int ndev = 0;
  AVH_CUDA_OK(cudaGetDeviceCount(&ndev));
  AVH_CHECK(device >= 0 && device < ndev, "no such CUDA device");
  cudaDeviceProp prop;
  AVH_CUDA_OK(cudaGetDeviceProperties(&prop, device));
  AVH_CHECK(prop.major == 10, "libavh_b200 contains sm_100a code only; this device is not a B200-class GPU");
  AVH_CUDA_OK(cudaSetDevice(device));
  avh_handle* h = new avh_handle();
  h->cfg = *cfg;
  h->device = device;
  h->P = cfg->compute_mode == AVH_COMPUTE_FP32 ? 2 : 1;
  *out = h;
  return 0;
}

int avh_destroy(avh_handle* h) {
  if (h == nullptr) return 0;
  cudaSetDevice(h->device);
  h->plans.clear();
  h->warena.release();
  for (auto& kv : h->staging) {
    if (kv.second.video) cudaFree(kv.second.video);
    if (kv.second.audio) cudaFree(kv.second.audio);
    if (kv.second.mask) cudaFree(kv.second.mask);
    if (kv.second.out) cudaFree(kv.second.out);
    if (kv.second.video_pp) cudaFree(kv.second.video_pp);
  }
  for (cudaEvent_t e : h->prof_events) cudaEventDestroy(e);
  if (h->refresh_exec) cudaGraphExecDestroy(h->refresh_exec);
  if (h->eval_refresh_exec) cudaGraphExecDestroy(h->eval_refresh_exec);
  delete h;
  return 0;
}

int avh_load_tensor(avh_handle* h, const char* key, const void* data, int dtype, const int64_t* shape, int ndim) {
  AVH_CHECK(h != nullptr && key != nullptr && data != nullptr, "null argument");
  AVH_CHECK(ndim >= 0 && ndim <= 8, "bad ndim");
  AVH_CHECK(dtype == AVH_F32 || dtype == AVH_F16 || dtype == AVH_BF16, "bad dtype");
  const std::string k(key);
  if (avh::ignorable_key(k)) return 0;
  AVH_CHECK(avh::known_prefix(k), "unexpected state-dict key: " + k);
  int64_t n = 1;
  for (int i = 0; i < ndim; ++i) n *= shape[i];
  AVH_CHECK(n >= 0 && n < (1ll << 31), "tensor too large");
  AVH_CUDA_OK(cudaSetDevice(h->device));
  std::vector<uint8_t> rawb((size_t)n * avh::dtype_size(dtype));
  AVH_CUDA_OK(cudaMemcpy(rawb.data(), data, rawb.size(), cudaMemcpyDefault));
  avh::HostTensor t;
  t.shape.assign(shape, shape + ndim);
  t.v.resize((size_t)n);
  if (dtype == AVH_F32) std::memcpy(t.v.data(), rawb.data(), rawb.size());
  else if (dtype == AVH_F16) {
    const __half* p = reinterpret_cast<const __half*>(rawb.data());
    for (int64_t i = 0; i < n; ++i) t.v[i] = __half2float(p[i]);
  } else {
    const __nv_bfloat16* p = reinterpret_cast<const __nv_bfloat16*>(rawb.data());
    for (int64_t i = 0; i < n; ++i) t.v[i] = __bfloat162float(p[i]);
  }
  h->raw[k] = std::move(t);
  h->finalized = false;
  return 0;
}

int avh_finalize_weights(avh_handle* h) {
  AVH_CHECK(h != nullptr, "null handle");
  AVH_CUDA_OK(cudaSetDevice(h->device));
  h->plans.clear();
  h->last_plan = nullptr;
  h->prof_plan = nullptr;
  h->warena.release();
  h->warena = avh::Arena();
  h->refresh_jobs.clear();
  if (h->refresh_exec) { cudaGraphExecDestroy(h->refresh_exec); h->refresh_exec = nullptr; }
  h->refresh_key.clear();
  h->eval_jobs.clear();
  if (h->eval_refresh_exec) { cudaGraphExecDestroy(h->eval_refresh_exec); h->eval_refresh_exec = nullptr; }
  h->eval_refresh_key.clear();
  avh::Packer sizer{h, nullptr, avh::Sizer(), ""};
  const bool ok = avh::pack_all(sizer);
  AVH_CHECK(ok, "missing state-dict key: " + sizer.missing);
  if (h->warena.init(sizer.sizer.used + (1 << 20))) return 1;
  avh::Packer pk{h, &h->warena, avh::Sizer(), ""};
  AVH_CHECK(avh::pack_all(pk), "weight upload failed");
  AVH_CHECK(h->warena.used <= h->warena.cap, "weight arena overflow");
  AVH_CUDA_OK(cudaDeviceSynchronize());
  h->finalized = true;
  return 0;
}

static int graphs_env = -1;      // 1 = CUDA-graph replay of the plan-internal runs of a launch list (AVH_GRAPHS=0: off)
static void read_graphs_env() {
  if (graphs_env >= 0) return;
  const char* ev = std::getenv("AVH_GRAPHS");
  const char* dbg = std::getenv("AVH_STEM_DBG");
  const char* dbg2 = std::getenv("AVH_WIN_DBG");
  graphs_env = ((ev != nullptr && ev[0] == '0') || dbg != nullptr || dbg2 != nullptr) ? 0 : 1;
}

// LayerDrop / modality dropout: a step of a dropped layer or modality arm is skipped and an on-drop step of a kept one;
// steps outside the layers and arms always run (plans without LayerDrop have an empty layer_skip, plans without modality
// dropout mod_drop 0)
static bool step_runs(const avh::Plan* p, const avh::Step& st) {
  const bool dropped = (st.layer >= 0 && st.layer < (int)p->layer_skip.size() && p->layer_skip[st.layer] != 0) ||
                       (st.mod != 0 && st.mod == p->mod_drop);
  return dropped == st.on_drop;
}

// capture every maximal run of plan-internal steps (they only enqueue kernels / async copies) into its own graph; in a
// plan with LayerDrop (modality dropout) a run also ends where the layer (modality arm) changes, so that a dropped
// layer's (arm's) graphs are skipped whole
static bool capture_segments(avh::Plan* p, cudaStream_t s) {
  bool ok = true;
  size_t i = 0;
  const bool by_layer = p->key.layerdrop, by_mod = p->key.moddrop;
  while (ok && i < p->steps.size()) {
    if (p->steps[i].direct) { ++i; continue; }
    size_t j = i;
    while (j < p->steps.size() && !p->steps[j].direct && (!by_layer || p->steps[j].layer == p->steps[i].layer) &&
           (!by_mod || p->steps[j].mod == p->steps[i].mod))
      ++j;
    const long long before = avh::g_launches.load();
    cudaGraph_t graph = nullptr;
    ok = cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
    if (ok) {
      for (size_t k = i; k < j; ++k)
        if (p->steps[k].run(s)) { ok = false; break; }
      if (cudaStreamEndCapture(s, &graph) != cudaSuccess || graph == nullptr) ok = false;
    }
    const int captured = (int)(avh::g_launches.load() - before);
    avh::count_launch(-captured);            // captured launches have not run
    cudaGraphExec_t exec = nullptr;
    if (ok && cudaGraphInstantiate(&exec, graph, 0) != cudaSuccess) ok = false;
    if (graph != nullptr) cudaGraphDestroy(graph);
    if (ok) p->segments.push_back(avh::Plan::Segment{i, j, exec, captured});
    i = j;
  }
  if (ok) p->segments_ready = true;
  else {
    // capture is not available for this launch list on this driver: remember, clear the error, run directly
    p->drop_graphs();
    cudaGetLastError();
    avh::g_err.clear();
    graphs_env = 0;
  }
  return ok;
}

// steps [begin, end) through the captured segments (direct steps launched in between); segments never straddle the range
static int replay_range(avh::Plan* p, size_t begin, size_t end, cudaStream_t s) {
  size_t i = begin, sg = 0;
  while (sg < p->segments.size() && p->segments[sg].begin < begin) ++sg;
  while (i < end) {
    if (sg < p->segments.size() && p->segments[sg].begin == i && p->segments[sg].end <= end) {
      if (step_runs(p, p->steps[i])) {      // a segment holds the steps of one layer (arm) when LayerDrop (modality dropout) is possible
        AVH_CUDA_OK(cudaGraphLaunch(p->segments[sg].exec, s));
        avh::count_launch(p->segments[sg].kernels);
        avh::g_graph_launches.fetch_add(1, std::memory_order_relaxed);
      }
      i = p->segments[sg].end;
      ++sg;
    } else {
      if (step_runs(p, p->steps[i]) && p->steps[i].run(s)) {
        if (avh::g_err.empty()) avh::set_last_error("kernel launch failed");
        return 1;
      }
      ++i;
    }
  }
  return 0;
}

// Steps [begin, end) of a plan: a whole forward, or the forward or backward half of a training plan.  The first run of
// a plan launches its steps directly (it also configures the kernels); the second captures every maximal run of
// plan-internal steps into a CUDA graph, later runs replay them (in a training plan the direct final-LayerNorm store
// separates the forward from the backward, so no graph straddles the two ranges).  The no-grad training-mode forward
// (its dropout seed is a launch argument) and profiled forwards always launch directly.  LayerDrop (step_runs) holds for
// every plan that has coins: direct runs and replays skip a dropped layer's steps alike.
static int run_steps(avh_handle* h, avh::Plan* p, size_t begin, size_t end, cudaStream_t s) {
  read_graphs_env();
  const avh::PlanKey& key = p->key;
  const bool train_fwd = key.kind == avh::PlanKind::TrainForward;
  const bool profiled = h->profiling && !key.training();     // avh_profile_json covers the forward plans
  // the caller's padding mask -> plan-owned copy (every later read is pointer-independent)
  if (begin == 0 && p->args.mask != nullptr)
    AVH_CUDA_OK(cudaMemcpyAsync(p->mask_dev, p->args.mask, (size_t)key.B * key.T, cudaMemcpyDeviceToDevice, s));
  // a caller that is itself capturing this stream (e.g. torch.cuda.graph) gets plain launches recorded into ITS graph
  cudaStreamCaptureStatus cap_status = cudaStreamCaptureStatusNone;
  if (s != nullptr && s != cudaStreamLegacy && s != cudaStreamPerThread) cudaStreamIsCapturing(s, &cap_status);
  const bool graphs_ok = graphs_env == 1 && !profiled && !train_fwd && s != nullptr && s != cudaStreamLegacy &&
                         s != cudaStreamPerThread && cap_status == cudaStreamCaptureStatusNone;
  if (graphs_ok && begin == 0 && !p->segments_ready && p->direct_runs >= 1) capture_segments(p, s);
  if (graphs_ok && graphs_env == 1 && p->segments_ready) return replay_range(p, begin, end, s);
  if (begin == 0) ++p->direct_runs;
  if (profiled) {
    while (h->prof_events.size() < 2 * p->steps.size()) {
      cudaEvent_t e;
      AVH_CUDA_OK(cudaEventCreate(&e));
      h->prof_events.push_back(e);
    }
    h->prof_plan = p;
  }
  for (size_t i = begin; i < end; ++i) {
    const avh::Step& st = p->steps[i];
    if (profiled) cudaEventRecord(h->prof_events[2 * i], s);
    if (step_runs(p, st) && st.run(s)) {
      if (avh::g_err.empty()) avh::set_last_error("kernel launch failed");
      return 1;
    }
    if (profiled) cudaEventRecord(h->prof_events[2 * i + 1], s);
  }
  return 0;
}

int avh_drop_host_weights(avh_handle* h) {
  AVH_CHECK(h != nullptr, "null handle");
  h->raw.clear();
  return 0;
}

int avh_release_stream(avh_handle* h, void* stream) {
  AVH_CHECK(h != nullptr, "null handle");
  AVH_CUDA_OK(cudaSetDevice(h->device));
  AVH_CUDA_OK(cudaStreamSynchronize(reinterpret_cast<cudaStream_t>(stream)));
  for (auto it = h->plans.begin(); it != h->plans.end();) {
    if (it->first.stream == reinterpret_cast<cudaStream_t>(stream)) {
      avh::forget_plan(h, it->second.get());
      it = h->plans.erase(it);
    } else ++it;
  }
  auto st = h->staging.find(stream);
  if (st != h->staging.end()) {
    void* ptrs[5] = {st->second.video, st->second.audio, st->second.mask, st->second.out, st->second.video_pp};
    for (void* q : ptrs)
      if (q) cudaFree(q);
    h->staging.erase(st);
  }
  return 0;
}

int avh_forward(avh_handle* h, const void* video, int video_dtype, const void* audio, int audio_dtype,
                const int64_t* audio_strides, const uint8_t* padding_mask, int B, int T, int output_layer,
                void* out, int out_dtype, void* stream) {
  AVH_CHECK(h != nullptr, "null handle");
  AVH_CHECK(h->finalized, "weights not finalized (call avh_finalize_weights)");
  AVH_CHECK(h->cfg.reserved[0] == 0, "this handle holds a bare TransformerEncoder: use avh_encoder_forward");
  AVH_CHECK(video != nullptr || audio != nullptr, "both modalities are None");
  AVH_CHECK(B >= 1 && T >= 1, "empty batch");
  AVH_CHECK((long long)B * T < (1ll << 24), "batch too large");
  AVH_CHECK(out != nullptr, "null output");
  AVH_CHECK(output_layer >= 0 && output_layer <= h->cfg.encoder_layers, "output_layer out of range");
  AVH_CHECK(audio == nullptr || audio_strides != nullptr, "audio strides required");
  AVH_CUDA_OK(cudaSetDevice(h->device));
  if (video != nullptr && video_dtype == AVH_U8) {
    // raw gray frames [B,1,T,src_h,src_w]: the dataset's /255 -> centre crop 88 -> (x-mean)/std on the device
    // (hubert_dataset.py:222-226; SURVEY 8(f)-1), into a per-stream buffer in the module's dtype
    avh_handle::Staging& st = h->staging[stream];
    const int pdt = h->cfg.compute_mode == AVH_COMPUTE_FP32 ? AVH_F32 : AVH_BF16;
    if (avh::ensure_cap(&st.video_pp, &st.video_pp_cap, (size_t)B * T * 7744 * avh::dtype_size(pdt))) return 1;
    if (avh::launch_video_preprocess(reinterpret_cast<const unsigned char*>(video), (long long)B * T, h->vp_src_h,
                                     h->vp_src_w, 88, h->vp_mean, h->vp_std, st.video_pp, pdt, padding_mask,
                                     reinterpret_cast<cudaStream_t>(stream)))
      return 1;
    video = st.video_pp;
    video_dtype = pdt;
  }
  AVH_CHECK(video == nullptr || video_dtype == AVH_F32 || video_dtype == AVH_F16 || video_dtype == AVH_BF16, "bad video dtype");
  avh::PlanKey key;
  key.kind = avh::PlanKind::Forward;
  key.B = B; key.T = T;
  key.has_video = video != nullptr; key.has_audio = audio != nullptr; key.has_mask = padding_mask != nullptr;
  key.output_layer = output_layer;
  key.stream = reinterpret_cast<cudaStream_t>(stream);
  avh::Plan* p = avh::get_plan(h, key);
  if (p == nullptr) return 1;
  h->last_plan = p;
  p->args.video = video; p->args.video_dt = video_dtype;
  p->args.audio = audio; p->args.audio_dt = audio_dtype;
  if (audio) for (int i = 0; i < 3; ++i) p->args.as[i] = audio_strides[i];
  p->args.mask = padding_mask;
  p->args.out = out; p->args.out_dt = out_dtype;
  return run_steps(h, p, 0, p->steps.size(), reinterpret_cast<cudaStream_t>(stream));
}

static int take_mod_drop(avh_handle* h, const void* video, const void* audio);

int avh_forward_train(avh_handle* h, const void* video, int video_dtype, const void* audio, int audio_dtype,
                      const int64_t* audio_strides, const uint8_t* padding_mask, int B, int T, int output_layer,
                      const avh_train_args* ta, void* out, int out_dtype, void* stream) {
  AVH_CHECK(h != nullptr && ta != nullptr, "null argument");
  AVH_CHECK(h->finalized, "weights not finalized (call avh_finalize_weights)");
  AVH_CHECK(h->cfg.reserved[0] == 0, "this handle holds a bare TransformerEncoder");
  AVH_CHECK(video != nullptr || audio != nullptr, "both modalities are None");
  AVH_CHECK(B >= 1 && T >= 1 && (long long)B * T < (1ll << 24), "bad batch");
  AVH_CHECK(out != nullptr, "null output");
  AVH_CHECK(output_layer >= 0 && output_layer <= h->cfg.encoder_layers, "output_layer out of range");
  AVH_CHECK(audio == nullptr || audio_strides != nullptr, "audio strides required");
  AVH_CHECK(video == nullptr || video_dtype == AVH_F32 || video_dtype == AVH_F16 || video_dtype == AVH_BF16,
            "training-mode forward takes normalised float video");
  AVH_CHECK(ta->attention_dropout == 0.f, "attention_dropout > 0 is not implemented (0.0 in every shipped fine-tune config)");
  for (float pr : {ta->dropout_input, ta->dropout, ta->activation_dropout})
    AVH_CHECK(pr >= 0.f && pr < 1.f, "dropout probabilities must be in [0, 1)");
  AVH_CHECK(ta->bn_momentum > 0.f && ta->bn_momentum <= 1.f, "bad BatchNorm momentum");
  AVH_CUDA_OK(cudaSetDevice(h->device));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int md = take_mod_drop(h, video, audio);
  if (md < -1) return 1;
  avh::PlanKey key;
  key.kind = avh::PlanKind::TrainForward;
  key.B = B; key.T = T;
  key.has_video = video != nullptr; key.has_audio = audio != nullptr; key.has_mask = padding_mask != nullptr;
  key.output_layer = output_layer;
  key.stream = s;
  key.moddrop = md >= 0;
  avh::Plan* p = avh::get_plan(h, key);
  if (p == nullptr) return 1;
  h->last_plan = p;
  p->mod_drop = md > 0 ? md : 0;
  p->args = avh::CallArgs();
  p->args.video = video; p->args.video_dt = video_dtype;
  p->args.audio = audio; p->args.audio_dt = audio_dtype;
  if (audio) for (int i = 0; i < 3; ++i) p->args.as[i] = audio_strides[i];
  p->args.mask = padding_mask;
  p->args.out = out; p->args.out_dt = out_dtype;
  p->p_in = ta->dropout_input; p->p_enc = ta->dropout; p->p_act = ta->activation_dropout;
  p->bn_momentum = ta->bn_momentum;
  p->seed = ta->seed;
  p->layer_skip.assign(h->cfg.encoder_layers, 0);
  if (ta->layer_skip != nullptr)
    for (int l = 0; l < h->cfg.encoder_layers; ++l) p->layer_skip[l] = ta->layer_skip[l];
  return run_steps(h, p, 0, p->steps.size(), s);
}

int avh_interp_linear(const void* x, int dtype, int B, int T, int C, const int32_t* len_in, const int32_t* len_out,
                      int Tout, void* out, int64_t* mask, void* stream) {
  AVH_CHECK(x != nullptr && out != nullptr && len_in != nullptr && len_out != nullptr, "null pointer");
  AVH_CHECK(dtype == AVH_F32 || dtype == AVH_F16 || dtype == AVH_BF16, "bad dtype");
  AVH_CHECK(B >= 1 && T >= 1 && C >= 1 && Tout >= 1, "bad shape");
  return avh::launch_interp_linear(x, dtype, B, T, C, len_in, len_out, Tout, out, reinterpret_cast<long long*>(mask),
                                   reinterpret_cast<cudaStream_t>(stream));
}

int avh_dropout(void* x, int dtype, int64_t n, float p, uint64_t seed, uint32_t site, void* stream) {
  AVH_CHECK(x != nullptr, "null pointer");
  AVH_CHECK(dtype == AVH_F32 || dtype == AVH_F16 || dtype == AVH_BF16, "bad dtype");
  return avh::launch_dropout(x, dtype, nullptr, n, p, seed, site, reinterpret_cast<cudaStream_t>(stream));
}

int avh_mask_substitute(const void* x, int dtype, int layout, const int64_t* strides, int B, int T, int U,
                        const int32_t* code, const void* emb, int emb_dtype, const uint8_t* channel_zero, void* out,
                        int out_dtype, void* stream) {
  AVH_CHECK(x != nullptr && code != nullptr && out != nullptr, "null pointer");
  AVH_CHECK(x != out, "mask substitution is out of place (sources are read from the un-substituted tensor)");
  AVH_CHECK(dtype == AVH_F32 || dtype == AVH_F16 || dtype == AVH_BF16, "bad dtype");
  AVH_CHECK(B >= 0 && T >= 0 && U > 0, "bad shape");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (layout == 0) {
    AVH_CHECK(out_dtype == dtype, "unit layout keeps the dtype");
    return avh::launch_mask_units(x, out, dtype, code, emb, emb_dtype, (long long)B * T, U, channel_zero, T, s);
  }
  AVH_CHECK(layout == 1, "layout must be 0 (contiguous units) or 1 (strided [B,C,T])");
  AVH_CHECK(strides != nullptr, "layout 1 needs the three element strides");
  AVH_CHECK(channel_zero == nullptr, "channel masks apply to the unit layout only");
  AVH_CHECK(out_dtype == AVH_F32 || out_dtype == AVH_F16 || out_dtype == AVH_BF16, "bad dtype");
  return avh::launch_mask_bct(x, dtype, strides[0], strides[1], strides[2], out, out_dtype, code, emb, emb_dtype, B, U, T, s);
}

int avh_compute_logits(const void* feats, int f_dtype, int64_t ldf, const void* emb, int e_dtype, int64_t lde,
                       const float* bias, int64_t M, int V, int K, int sim_type, float logit_temp, float* out, int64_t ldo,
                       void* stream) {
  AVH_CHECK(feats != nullptr && emb != nullptr && out != nullptr, "null pointer");
  AVH_CHECK(sim_type == 0 || sim_type == 1, "sim_type must be 0 (dot) or 1 (cosine)");
  AVH_CHECK(logit_temp != 0.f, "logit_temp must be non-zero");
  AVH_CHECK(K > 0 && ldf >= K && lde >= K && ldo >= V, "bad leading dimension");
  return avh::launch_logits(feats, f_dtype, ldf, emb, e_dtype, lde, bias, out, ldo, M, V, K, sim_type, 1.0f / logit_temp,
                            reinterpret_cast<cudaStream_t>(stream));
}

int avh_sum_squares(const void* x, int dtype, int64_t n, double* acc, void* stream) {
  AVH_CHECK(x != nullptr && acc != nullptr, "null pointer");
  return avh::launch_sumsq(x, dtype, n, acc, reinterpret_cast<cudaStream_t>(stream));
}

int avh_compute_logits_backward(const void* feats, int f_dtype, int64_t ldf, const void* emb, int e_dtype, int64_t lde, int64_t M,
                                int V, int K, int sim_type, float logit_temp, const float* logits, const float* dlogits,
                                int64_t ldo, float* dfeats, int64_t ldd_f, float* demb, int64_t ldd_e, float* dbias, void* stream) {
  AVH_CHECK(feats != nullptr && emb != nullptr && dlogits != nullptr, "null pointer");
  AVH_CHECK(sim_type == 0 || sim_type == 1, "sim_type must be 0 (dot) or 1 (cosine)");
  AVH_CHECK(sim_type == 0 || logits != nullptr, "the cosine backward reads the forward's logits");
  AVH_CHECK(logit_temp != 0.f, "logit_temp must be non-zero");
  AVH_CHECK(M >= 0 && V >= 0 && K > 0 && ldf >= K && lde >= K && ldo >= V, "bad leading dimension");
  AVH_CHECK((dfeats == nullptr || ldd_f >= K) && (demb == nullptr || ldd_e >= K), "bad gradient leading dimension");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  float* scratch = nullptr;      // norms, row / column sums, split-contraction partials: stream-ordered, freed after use
  if (M > 0 && V > 0)
    AVH_CUDA_OK(cudaMallocAsync(reinterpret_cast<void**>(&scratch), (size_t)avh::logits_bwd_scratch_floats(M, V, K) * sizeof(float), s));
  const int rc = avh::launch_logits_bwd(feats, f_dtype, ldf, emb, e_dtype, lde, M, V, K, sim_type, 1.0f / logit_temp, logits, dlogits,
                                        ldo, dfeats, ldd_f, demb, ldd_e, dbias, scratch, s);
  if (scratch != nullptr) AVH_CUDA_OK(cudaFreeAsync(scratch, s));
  return rc;
}

int avh_set_modality_drop(avh_handle* h, int which) {
  AVH_CHECK(h != nullptr && h->cfg.reserved[0] == 0, "modality dropout belongs to an AV-HuBERT handle");
  AVH_CHECK(which >= 0 && which <= 2, "which must be 0 (none), 1 (audio) or 2 (video)");
  h->next_mod_drop = which;
  return 0;
}

// The pending avh_set_modality_drop decision (consumed): -1 = not a pretraining step
static int take_mod_drop(avh_handle* h, const void* video, const void* audio) {
  const int md = h->next_mod_drop;
  h->next_mod_drop = -1;
  if (md >= 0 && (video == nullptr || audio == nullptr)) {
    avh::set_last_error("modality dropout needs both modalities");
    return -2;
  }
  return md;
}

int avh_train_features_pen(avh_handle* h, double* acc, void* stream) {
  AVH_CHECK(h != nullptr && acc != nullptr, "null argument");
  const avh::Plan* p = h->last_plan;
  AVH_CHECK(p != nullptr && (p->key.kind == avh::PlanKind::TrainForward || p->key.training()) && p->fused_buf != nullptr,
            "features_pen follows a training-mode forward of an AV-HuBERT handle");
  AVH_CUDA_OK(cudaSetDevice(h->device));
  const int E = h->cfg.modality_fuse == AVH_FUSE_CONCAT ? 2 * h->cfg.encoder_embed_dim : h->cfg.encoder_embed_dim;
  return avh::launch_sumsq(p->fused_buf, p->fused_dt, (long long)p->key.B * p->key.T * E, acc, reinterpret_cast<cudaStream_t>(stream));
}

int avh_set_features_pen_grad(avh_handle* h, const float* dpen, void* stream) {
  AVH_CHECK(h != nullptr, "null handle");
  avh::Plan* p = h->last_plan;
  AVH_CHECK(p != nullptr && p->dpen != nullptr && p->fwd_done,
            "the features_pen gradient belongs to a pretraining avh_full_train_forward (avh_set_modality_drop first)");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  AVH_CHECK(s == p->key.stream, "the features_pen gradient must be set on the stream of its forward");
  AVH_CUDA_OK(cudaSetDevice(h->device));
  if (dpen != nullptr) AVH_CUDA_OK(cudaMemcpyAsync(p->dpen, dpen, sizeof(float), cudaMemcpyDeviceToDevice, s));
  else AVH_CUDA_OK(cudaMemsetAsync(p->dpen, 0, sizeof(float), s));
  return 0;
}

int avh_bn_stats_count(avh_handle* h, int64_t* n_floats) {
  AVH_CHECK(h != nullptr && n_floats != nullptr, "null argument");
  AVH_CHECK(h->finalized, "weights not finalized");
  int64_t n = 2 * 64;
  for (int L = 0; L < 4; ++L)
    for (int bi = 0; bi < 2; ++bi) n += 2 * (64 << L) * (h->blocks[L][bi].has_ds ? 3 : 2);
  *n_floats = n;
  return 0;
}

int avh_read_bn_stats(avh_handle* h, float* dst, int64_t capacity, void* stream) {
  AVH_CHECK(h != nullptr && dst != nullptr, "null argument");
  AVH_CHECK(h->finalized && h->cfg.reserved[0] == 0, "no lip frontend in this handle");
  int64_t need = 0;
  if (avh_bn_stats_count(h, &need)) return 1;
  AVH_CHECK(capacity >= need, "destination too small");
  AVH_CUDA_OK(cudaSetDevice(h->device));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  int64_t off = 0;
  auto put = [&](const avh::ConvUnit& cu, int C) -> int {
    AVH_CUDA_OK(cudaMemcpyAsync(dst + off, cu.rmean, (size_t)C * 4, cudaMemcpyDeviceToDevice, s));
    AVH_CUDA_OK(cudaMemcpyAsync(dst + off + C, cu.rvar, (size_t)C * 4, cudaMemcpyDeviceToDevice, s));
    off += 2 * C;
    return 0;
  };
  if (put(h->stem, 64)) return 1;
  for (int L = 0; L < 4; ++L)
    for (int bi = 0; bi < 2; ++bi) {
      const avh::BlockW& bw = h->blocks[L][bi];
      if (put(bw.c1, 64 << L) || put(bw.c2, 64 << L)) return 1;
      if (bw.has_ds && put(bw.ds, 64 << L)) return 1;
    }
  return 0;
}

int avh_encoder_forward(avh_handle* h, const void* x, int x_dtype, const uint8_t* padding_mask, int B, int T,
                        int output_layer, void* out, int out_dtype, void* stream) {
  AVH_CHECK(h != nullptr, "null handle");
  AVH_CHECK(h->finalized, "weights not finalized (call avh_finalize_weights)");
  AVH_CHECK(x != nullptr && out != nullptr, "null argument");
  AVH_CHECK(x_dtype == AVH_F32 || x_dtype == AVH_F16 || x_dtype == AVH_BF16, "bad feature dtype");
  AVH_CHECK(h->cfg.reserved[0] != 2, "this handle holds a Q-Former: use avh_qformer_forward");
  AVH_CHECK(B >= 1 && T >= 1 && (long long)B * T < (1ll << 24), "bad batch");
  AVH_CHECK(output_layer >= 0 && output_layer <= h->cfg.encoder_layers, "output_layer out of range");
  AVH_CUDA_OK(cudaSetDevice(h->device));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  avh::PlanKey key;
  key.kind = avh::PlanKind::EncoderOnly;
  key.B = B; key.T = T;
  key.has_mask = padding_mask != nullptr;
  key.output_layer = output_layer;
  key.stream = s;
  avh::Plan* p = avh::get_plan(h, key);
  if (p == nullptr) return 1;
  h->last_plan = p;
  p->args = avh::CallArgs();
  p->args.xin = x; p->args.xin_dt = x_dtype;
  p->args.mask = padding_mask;
  p->args.out = out; p->args.out_dt = out_dtype;
  return run_steps(h, p, 0, p->steps.size(), s);
}

int avh_encoder_grad_count(avh_handle* h, int64_t* n_floats) {
  AVH_CHECK(h != nullptr && n_floats != nullptr, "null argument");
  AVH_CHECK(h->cfg.reserved[0] != 2, "this handle holds a Q-Former");
  *n_floats = avh::enc_grad_floats(h->cfg);
  return 0;
}

static int encoder_train_forward(avh_handle* h, const void* x, int x_dtype, const uint8_t* padding_mask, int B, int T, void* out,
                                 int out_dtype, void* stream, bool tail);

int avh_set_train_args(avh_handle* h, const avh_train_args* ta) {
  AVH_CHECK(h != nullptr && ta != nullptr, "null argument");
  AVH_CHECK(ta->attention_dropout == 0.f, "attention_dropout > 0 is not implemented (0.0 in every shipped fine-tune config)");
  for (float pr : {ta->dropout_input, ta->dropout, ta->activation_dropout})
    AVH_CHECK(pr >= 0.f && pr < 1.f, "dropout probabilities must be in [0, 1)");
  avh_handle::NextTrain nt;
  nt.p_in = ta->dropout_input; nt.p_enc = ta->dropout; nt.p_act = ta->activation_dropout;
  nt.seed = ta->seed;
  if (ta->layer_skip != nullptr) nt.skip.assign(ta->layer_skip, ta->layer_skip + h->cfg.encoder_layers);
  h->next_train = std::move(nt);
  return 0;
}

// The plan of a training step with the regularisation avh_set_train_args left for it (consumed here; none: a plain
// step): probabilities and "LayerDrop possible" select the plan, the seed goes to its device word and the coins to its
// layer_skip, which the backward of this step reads too.  site1: the plan has dropout_input (tail modes).
static avh::Plan* training_plan(avh_handle* h, avh::PlanKey key, bool site1, cudaStream_t s) {
  avh_handle::NextTrain nt = std::move(h->next_train);
  h->next_train = avh_handle::NextTrain();
  key.p_in = site1 ? nt.p_in : 0.f;
  key.p_enc = nt.p_enc;
  key.p_act = nt.p_act;
  key.layerdrop = !nt.skip.empty();
  avh::Plan* p = avh::get_plan(h, key);
  if (p == nullptr) return nullptr;
  p->layer_skip = std::move(nt.skip);
  if (p->seed_dev != nullptr) {
    const int slot = p->seed_next;
    p->seed_next = (slot + 1) % avh::Plan::RAG_SLOTS;
    cudaError_t e = cudaEventSynchronize(p->seed_done[slot]);      // the copy that last read this mirror has run
    if (e == cudaSuccess) {
      *p->seed_host[slot] = nt.seed;
      e = cudaMemcpyAsync(p->seed_dev, p->seed_host[slot], sizeof(unsigned long long), cudaMemcpyHostToDevice, s);
    }
    if (e == cudaSuccess) e = cudaEventRecord(p->seed_done[slot], s);
    if (e != cudaSuccess) {
      avh::set_last_error(std::string("dropout seed upload failed: ") + cudaGetErrorString(e));
      return nullptr;
    }
  }
  return p;
}

int avh_tail_grad_count(avh_handle* h, int64_t* n_floats) {
  AVH_CHECK(h != nullptr && n_floats != nullptr, "null argument");
  AVH_CHECK(h->cfg.reserved[0] == 0, "the trainable tail belongs to an AV-HuBERT handle");
  *n_floats = avh::enc_grad_floats(h->cfg, true);
  return 0;
}

int avh_tail_train_forward(avh_handle* h, const void* fused, int dtype, const uint8_t* padding_mask, int B, int T, void* out,
                           int out_dtype, void* stream) {
  AVH_CHECK(h != nullptr && h->cfg.reserved[0] == 0, "the trainable tail belongs to an AV-HuBERT handle");
  return encoder_train_forward(h, fused, dtype, padding_mask, B, T, out, out_dtype, stream, true);
}

int avh_encoder_train_forward(avh_handle* h, const void* x, int x_dtype, const uint8_t* padding_mask, int B, int T, void* out,
                              int out_dtype, void* stream) {
  return encoder_train_forward(h, x, x_dtype, padding_mask, B, T, out, out_dtype, stream, false);
}

int avh_full_grad_count(avh_handle* h, int has_video, int has_audio, int64_t* n_floats) {
  AVH_CHECK(h != nullptr && n_floats != nullptr, "null argument");
  AVH_CHECK(h->cfg.reserved[0] == 0, "the full training step belongs to an AV-HuBERT handle");
  *n_floats = avh::enc_grad_floats(h->cfg, 2, has_video != 0, has_audio != 0);
  return 0;
}

int avh_full_train_forward(avh_handle* h, const void* video, int video_dtype, const void* audio, int audio_dtype,
                           const int64_t* audio_strides, const uint8_t* padding_mask, int B, int T, float feature_grad_mult,
                           float bn_momentum, void* out, int out_dtype, void* stream) {
  AVH_CHECK(h != nullptr, "null handle");
  AVH_CHECK(h->finalized, "weights not finalized (call avh_finalize_weights)");
  AVH_CHECK(h->cfg.reserved[0] == 0, "the full training step belongs to an AV-HuBERT handle");
  AVH_CHECK(h->cfg.reserved[3] != 0, "handle not created as trainable (avh_config.reserved[3] = 1)");
  AVH_CHECK(video != nullptr || audio != nullptr, "both modalities are None");
  AVH_CHECK(out != nullptr, "null argument");
  AVH_CHECK(video == nullptr || video_dtype == AVH_F32 || video_dtype == AVH_F16 || video_dtype == AVH_BF16,
            "the training step takes normalised float video");
  AVH_CHECK(audio == nullptr || audio_strides != nullptr, "audio strides required");
  AVH_CHECK(B >= 1 && T >= 1 && (long long)B * T < (1ll << 20), "bad batch");
  AVH_CUDA_OK(cudaSetDevice(h->device));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int md = take_mod_drop(h, video, audio);
  if (md < -1) return 1;
  avh::PlanKey key;
  key.kind = avh::PlanKind::FullTrain;
  key.B = B; key.T = T;
  key.has_video = video != nullptr; key.has_audio = audio != nullptr; key.has_mask = padding_mask != nullptr;
  key.stream = s;
  key.moddrop = key.pen = md >= 0;
  avh::Plan* p = training_plan(h, key, true, s);
  if (p == nullptr) return 1;
  h->last_plan = p;
  p->mod_drop = md > 0 ? md : 0;
  if (p->dpen != nullptr) AVH_CUDA_OK(cudaMemsetAsync(p->dpen, 0, sizeof(float), s));      // no dL/dpen unless set
  p->args = avh::CallArgs();
  p->args.video = video; p->args.video_dt = video_dtype;
  p->args.audio = audio; p->args.audio_dt = audio_dtype;
  if (audio) for (int i = 0; i < 3; ++i) p->args.as[i] = audio_strides[i];
  p->args.mask = padding_mask;
  p->args.out = out; p->args.out_dt = out_dtype;
  p->bn_momentum = bn_momentum;
  p->fgm = feature_grad_mult;
  p->fwd_done = false;
  if (run_steps(h, p, 0, p->fwd_steps, s)) return 1;
  p->fwd_done = true;
  return 0;
}

static int encoder_train_forward(avh_handle* h, const void* x, int x_dtype, const uint8_t* padding_mask, int B, int T, void* out,
                                 int out_dtype, void* stream, bool tail) {
  AVH_CHECK(h != nullptr, "null handle");
  AVH_CHECK(h->finalized, "weights not finalized (call avh_finalize_weights)");
  AVH_CHECK(h->cfg.reserved[0] != 2, "this handle holds a Q-Former");
  AVH_CHECK(h->cfg.reserved[3] != 0, "handle not created as trainable (avh_config.reserved[3] = 1 packs the backward's operands)");
  AVH_CHECK(x != nullptr && out != nullptr, "null argument");
  AVH_CHECK(x_dtype == AVH_F32 || x_dtype == AVH_F16 || x_dtype == AVH_BF16, "bad feature dtype");
  AVH_CHECK(B >= 1 && T >= 1 && (long long)B * T < (1ll << 24), "bad batch");
  AVH_CUDA_OK(cudaSetDevice(h->device));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  avh::PlanKey key;
  key.kind = tail ? avh::PlanKind::TailTrain : avh::PlanKind::EncoderTrain;
  key.B = B; key.T = T;
  key.has_mask = padding_mask != nullptr;
  key.stream = s;
  avh::Plan* p = training_plan(h, key, tail, s);
  if (p == nullptr) return 1;
  h->last_plan = p;
  p->args = avh::CallArgs();
  p->args.xin = x; p->args.xin_dt = x_dtype;
  p->args.mask = padding_mask;
  p->args.out = out; p->args.out_dt = out_dtype;
  p->fwd_done = false;
  if (run_steps(h, p, 0, p->fwd_steps, s)) return 1;
  p->fwd_done = true;
  return 0;
}

// The backward half of the last training plan.  `buckets`: the gradient buckets are converted into the caller's `grads`
// (of dtype grads_dtype) as the backward completes them; otherwise the whole fp32 buffer is copied at the end, if asked.
static int encoder_backward(avh_handle* h, const void* dout, int dout_dtype, void* dx, int dx_dtype, void* grads, int grads_dtype,
                            int64_t grads_capacity, bool buckets, void* stream) {
  AVH_CHECK(h != nullptr, "null handle");
  AVH_CHECK(dout != nullptr && (grads != nullptr || !buckets), "null argument");
  AVH_CHECK(!buckets || grads_dtype == AVH_F32 || grads_dtype == AVH_BF16 || grads_dtype == AVH_F16, "bad gradient dtype");
  avh::Plan* p = h->last_plan;
  AVH_CHECK(p != nullptr && p->key.training() && p->fwd_done, "the backward follows a training forward on the same handle");
  AVH_CHECK(grads == nullptr || grads_capacity >= p->grad_floats, "gradient buffer too small (avh_encoder_grad_count)");
  AVH_CUDA_OK(cudaSetDevice(h->device));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  AVH_CHECK(s == p->key.stream, "backward must run on the stream of its forward");
  const long long N = (long long)p->key.B * p->key.T;
  const int D = h->cfg.encoder_embed_dim;
  // dL/dy -> fp32.  Rows of padded frames are taken as given, as autograd does: the dense forward computed those rows
  // (their queries attend to the valid keys), so a loss that reads them sends gradient through them too
  if (avh::launch_load_rows(dout, dout_dtype, p->dy_in, nullptr, N, D, s)) return 1;
  p->args.grads_out = buckets ? grads : nullptr;
  p->args.grads_dt = grads_dtype;
  const int rc = run_steps(h, p, p->fwd_steps, p->steps.size(), s);
  p->args.grads_out = nullptr;
  if (rc) return 1;
  if (dx != nullptr && avh::launch_convert(p->dx_out, avh::DT_F32, dx, dx_dtype, N * D, s)) return 1;
  if (!buckets && grads != nullptr)
    AVH_CUDA_OK(cudaMemcpyAsync(grads, p->grads, (size_t)p->grad_floats * 4, cudaMemcpyDeviceToDevice, s));
  p->fwd_done = false;
  return 0;
}

int avh_encoder_backward(avh_handle* h, const void* dout, int dout_dtype, void* dx, int dx_dtype, float* grads,
                         int64_t grads_capacity, void* stream) {
  return encoder_backward(h, dout, dout_dtype, dx, dx_dtype, grads, AVH_F32, grads_capacity, false, stream);
}

int avh_encoder_backward_buckets(avh_handle* h, const void* dout, int dout_dtype, void* dx, int dx_dtype, void* grads,
                                 int grads_dtype, int64_t grads_capacity, void* stream) {
  return encoder_backward(h, dout, dout_dtype, dx, dx_dtype, grads, grads_dtype, grads_capacity, true, stream);
}

// The caller's tensor list of a device refresh: state-dict key -> index, and the pointer set the captured graph is keyed on
struct RefreshArgs {
  std::map<std::string, int> idx;
  const void* const* ptrs = nullptr;
  const int32_t* dtypes = nullptr;
  const int64_t* numels = nullptr;
  std::vector<long long> key;
};

static int refresh_args(const char* const* names, const void* const* ptrs, const int32_t* dtypes, const int64_t* numels,
                        int32_t count, RefreshArgs* a) {
  AVH_CHECK(names != nullptr && ptrs != nullptr && dtypes != nullptr && numels != nullptr, "null argument");
  for (int i = 0; i < count; ++i) {
    AVH_CHECK(names[i] != nullptr && ptrs[i] != nullptr, "null tensor in the parameter list");
    AVH_CHECK(dtypes[i] == AVH_F32 || dtypes[i] == AVH_F16 || dtypes[i] == AVH_BF16, "bad parameter dtype");
    a->idx[names[i]] = i;
  }
  a->ptrs = ptrs; a->dtypes = dtypes; a->numels = numels;
  a->key.reserve(3 * (size_t)count);
  for (int i = 0; i < count; ++i) {
    a->key.push_back((long long)reinterpret_cast<uintptr_t>(ptrs[i]));
    a->key.push_back(dtypes[i]);
    a->key.push_back(numels[i]);
  }
  return 0;
}

// the training-form jobs (refresh_jobs; empty on handles that are not trainable)
static int run_train_refresh(avh_handle* h, const RefreshArgs& a, cudaStream_t s) {
  const int P = h->P;
  const int KT = h->cfg.conv_pos;
  bool ratio_done = false;
  for (const avh_handle::RefreshJob& j : h->refresh_jobs) {
    auto it = a.idx.find(j.src);
    AVH_CHECK(it != a.idx.end(), "parameter missing from the refresh list: " + j.src);
    const int i = it->second;
    const void* src = a.ptrs[i];
    const int dt = a.dtypes[i];
    const long long ne = a.numels[i];
    switch (j.form) {
      case avh::RJ_MATRIX:
      case avh::RJ_MATRIX_T:
        AVH_CHECK(ne == j.n * j.k, "parameter size changed: " + j.src);
        if (avh::launch_refresh_matrix(src, dt, j.n, j.k, j.scale, j.dst, j.ld, P, j.off, j.form == avh::RJ_MATRIX_T, s)) return 1;
        break;
      case avh::RJ_VEC:
      case avh::RJ_VEC_OFF:
        AVH_CHECK(ne == j.n || ne == 1, "parameter size changed: " + j.src);
        if (avh::launch_refresh_vec(src, dt, j.n, ne, j.scale, reinterpret_cast<float*>(j.dst) + j.off, s)) return 1;
        break;
      case avh::RJ_CONV:
      case avh::RJ_CONV_T:
        AVH_CHECK(ne == j.n * j.k * j.ks * j.ks, "parameter size changed: " + j.src);
        if (avh::launch_refresh_conv(src, dt, (int)j.n, (int)j.k, j.ks * j.ks, j.dst, j.ld, P, j.form == avh::RJ_CONV_T, s)) return 1;
        break;
      case avh::RJ_STEM:
        AVH_CHECK(ne == 64 * 245, "parameter size changed: " + j.src);
        if (avh::launch_refresh_stem(src, dt, j.dst, P, j.ks == 8 ? 1 : 0, s)) return 1;
        break;
      case avh::RJ_POS:
      case avh::RJ_POS_T: {
        AVH_CHECK(ne == j.n * j.k * KT && h->pos_ratio != nullptr, "parameter size changed: " + j.src);
        if (!ratio_done) {
          auto ig = a.idx.find("encoder.pos_conv.0.weight_g");
          AVH_CHECK(ig != a.idx.end() && a.numels[ig->second] == KT, "parameter missing from the refresh list: encoder.pos_conv.0.weight_g");
          if (avh::launch_posconv_ratio(src, dt, a.ptrs[ig->second], a.dtypes[ig->second], j.n * j.k, KT, h->pos_ratio, s)) return 1;
          ratio_done = true;
        }
        if (avh::launch_refresh_pos(src, dt, h->pos_ratio, h->pos_acol, (int)j.n, (int)j.k, KT, h->pos_window, j.dst, P,
                                    j.form == avh::RJ_POS_T, s))
          return 1;
        break;
      }
      default:
        AVH_CHECK(false, "unknown refresh job");
    }
  }
  return 0;
}

// the eval-only forms (eval_jobs): BatchNorm folds, then the conv2 + shortcut GEMM weights that read them
static int run_eval_refresh(avh_handle* h, const RefreshArgs& a, cudaStream_t s) {
  auto find = [&](const std::string& key, long long numel, int* i) -> int {
    auto it = a.idx.find(key);
    AVH_CHECK(it != a.idx.end(), "tensor missing from the refresh list: " + key);
    AVH_CHECK(a.numels[it->second] == numel, "tensor size changed: " + key);
    *i = it->second;
    return 0;
  };
  for (const avh_handle::EvalJob& j : h->eval_jobs) {
    if (j.bw == nullptr) {
      ConvUnit* cu = j.cu;
      const char* part[4] = {".weight", ".bias", ".running_mean", ".running_var"};
      int i[4];
      for (int t = 0; t < 4; ++t)
        if (find(j.bn + part[t], cu->cout, &i[t])) return 1;
      if (avh::launch_bn_fold(a.ptrs[i[0]], a.dtypes[i[0]], a.ptrs[i[1]], a.dtypes[i[1]], a.ptrs[i[2]], a.dtypes[i[2]], a.ptrs[i[3]],
                              a.dtypes[i[3]], cu->cout, cu->scale, cu->bias, cu->gamma, cu->beta, cu->rmean, cu->rvar, s))
        return 1;
    } else {
      const BlockW* bw = j.bw;
      const int cout = bw->c2.cout, cmid = bw->c2.cin, cin = bw->ds.cin;
      int i2, id;
      if (find(j.w2, 9LL * cout * cmid, &i2) || find(j.wd, (long long)cout * cin, &id)) return 1;
      if (avh::launch_refresh_c2ds(a.ptrs[i2], a.dtypes[i2], a.ptrs[id], a.dtypes[id], bw->c2.scale, bw->c2.bias, bw->ds.scale,
                                   bw->ds.bias, cout, cmid, cin, bw->c2ds.w, h->P, bw->c2ds_bias, s))
        return 1;
    }
  }
  return 0;
}

// Runs `jobs` on `s` through a CUDA graph captured for the pointer set `key` (an optimizer updates the same tensors in
// place every step: hundreds of small launches become one graph launch); `*exec` / `*exec_key` cache the graph.  Directly
// where the stream cannot be captured (the legacy default stream).
static int replay_refresh(cudaStream_t s, const std::vector<long long>& key, cudaGraphExec_t* exec, std::vector<long long>* exec_key,
                          const std::function<int()>& jobs) {
  if (*exec != nullptr && key == *exec_key) {
    AVH_CUDA_OK(cudaGraphLaunch(*exec, s));
    return 0;
  }
  if (*exec) { cudaGraphExecDestroy(*exec); *exec = nullptr; }
  exec_key->clear();
  read_graphs_env();
  cudaStreamCaptureStatus cap_status = cudaStreamCaptureStatusNone;
  const bool real_stream = s != nullptr && s != cudaStreamLegacy && s != cudaStreamPerThread;
  if (real_stream) cudaStreamIsCapturing(s, &cap_status);
  if (graphs_env == 1 && real_stream && cap_status == cudaStreamCaptureStatusNone &&
      cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
    const int rc = jobs();
    cudaGraph_t graph = nullptr;
    const cudaError_t e = cudaStreamEndCapture(s, &graph);
    cudaGraphExec_t ex = nullptr;
    const bool ok = rc == 0 && e == cudaSuccess && graph != nullptr && cudaGraphInstantiate(&ex, graph, 0) == cudaSuccess;
    if (graph != nullptr) cudaGraphDestroy(graph);
    if (rc != 0) return 1;                         // a real error (missing / resized parameter): reported as is
    if (ok) {
      *exec = ex;
      *exec_key = key;
      AVH_CUDA_OK(cudaGraphLaunch(ex, s));
      return 0;
    }
  }
  cudaGetLastError();                              // capture not possible on this stream (legacy default stream): direct
  return jobs();
}

int avh_refresh_weights_device(avh_handle* h, const char* const* names, const void* const* ptrs, const int32_t* dtypes,
                               const int64_t* numels, int32_t count, void* stream) {
  AVH_CHECK(h != nullptr, "null argument");
  AVH_CHECK(h->finalized, "weights not finalized (call avh_finalize_weights once; this call refreshes them in place)");
  AVH_CHECK(h->cfg.reserved[3] != 0, "only trainable handles (avh_config.reserved[3] = 1) record how to refresh their weights");
  AVH_CUDA_OK(cudaSetDevice(h->device));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  RefreshArgs a;
  if (refresh_args(names, ptrs, dtypes, numels, count, &a)) return 1;
  return replay_refresh(s, a.key, &h->refresh_exec, &h->refresh_key, [&]() { return run_train_refresh(h, a, s); });
}

int avh_refresh_eval_weights_device(avh_handle* h, const char* const* names, const void* const* ptrs, const int32_t* dtypes,
                                    const int64_t* numels, int32_t count, void* stream) {
  AVH_CHECK(h != nullptr, "null argument");
  AVH_CHECK(h->finalized, "weights not finalized (call avh_finalize_weights once; this call refreshes them in place)");
  AVH_CHECK(h->cfg.reserved[0] != 2, "Q-Former handles have no device refresh (reload the weights and finalize)");
  AVH_CUDA_OK(cudaSetDevice(h->device));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  RefreshArgs a;
  if (refresh_args(names, ptrs, dtypes, numels, count, &a)) return 1;
  return replay_refresh(s, a.key, &h->eval_refresh_exec, &h->eval_refresh_key,
                        [&]() { return run_train_refresh(h, a, s) || run_eval_refresh(h, a, s) ? 1 : 0; });
}

int avh_plan_count(avh_handle* h, int32_t* count) {
  AVH_CHECK(h != nullptr && count != nullptr, "null argument");
  *count = (int32_t)h->plans.size();
  return 0;
}

int avh_grad_bucket_count(avh_handle* h, int32_t* count) {
  AVH_CHECK(h != nullptr && count != nullptr, "null argument");
  avh::Plan* p = h->last_plan;
  AVH_CHECK(p != nullptr && p->key.training(), "no training plan on this handle yet (run a training forward first)");
  *count = (int32_t)p->buckets.size();
  return 0;
}

int avh_grad_bucket_range(avh_handle* h, int k, int64_t* begin, int64_t* end) {
  AVH_CHECK(h != nullptr && begin != nullptr && end != nullptr, "null argument");
  avh::Plan* p = h->last_plan;
  AVH_CHECK(p != nullptr && p->key.training() && k >= 0 && k < (int)p->buckets.size(), "bucket index out of range");
  *begin = p->buckets[k].begin;
  *end = p->buckets[k].end;
  return 0;
}

int avh_grad_bucket_wait(avh_handle* h, int k, void* stream) {
  AVH_CHECK(h != nullptr, "null handle");
  avh::Plan* p = h->last_plan;
  AVH_CHECK(p != nullptr && p->key.training() && k >= 0 && k < (int)p->buckets.size(), "bucket index out of range");
  AVH_CUDA_OK(cudaSetDevice(h->device));
  AVH_CUDA_OK(cudaStreamWaitEvent(reinterpret_cast<cudaStream_t>(stream), p->buckets[k].ev, 0));
  return 0;
}

int avh_qformer_forward(avh_handle* h, const void* enc, int enc_dtype, const uint8_t* enc_padding, const int32_t* len_queries,
                        int B, int Lq, int Lk, void* out, int out_dtype, void* stream) {
  AVH_CHECK(h != nullptr, "null handle");
  AVH_CHECK(h->cfg.reserved[0] == 2, "this handle does not hold a Q-Former");
  AVH_CHECK(h->finalized, "weights not finalized (call avh_finalize_weights)");
  AVH_CHECK(enc != nullptr && out != nullptr, "null argument");
  AVH_CHECK(enc_dtype == AVH_F32 || enc_dtype == AVH_F16 || enc_dtype == AVH_BF16, "bad feature dtype");
  AVH_CHECK(B >= 1 && Lq >= 1 && Lk >= 1 && (long long)B * Lk < (1ll << 24), "bad batch");
  AVH_CHECK(Lq <= h->cfg.reserved[2], "more queries than query_tokens holds");
  AVH_CUDA_OK(cudaSetDevice(h->device));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  avh::PlanKey key;
  key.kind = avh::PlanKind::QFormer;
  key.B = B; key.T = Lq; key.Lk = Lk;
  key.has_mask = enc_padding != nullptr;
  key.stream = s;
  avh::Plan* p = avh::get_plan(h, key);
  if (p == nullptr) return 1;
  h->last_plan = p;
  // query attention mask (src/model.py:588-590): row i of clip b is a key for the queries iff i < len_queries[b]
  std::vector<unsigned char> qm((size_t)B * Lq, 0);
  if (len_queries != nullptr)
    for (int b = 0; b < B; ++b) {
      AVH_CHECK(len_queries[b] >= 1 && len_queries[b] <= Lq, "len_queries must be in [1, Lq]");
      for (int i = len_queries[b]; i < Lq; ++i) qm[(size_t)b * Lq + i] = 1;
    }
  AVH_CUDA_OK(cudaMemcpyAsync(p->qmask_dev, qm.data(), qm.size(), cudaMemcpyHostToDevice, s));      // pageable: staged before return
  if (enc_padding != nullptr)
    AVH_CUDA_OK(cudaMemcpyAsync(p->kmask_dev, enc_padding, (size_t)B * Lk, cudaMemcpyDeviceToDevice, s));
  p->args = avh::CallArgs();
  p->args.xin = enc; p->args.xin_dt = enc_dtype;
  p->args.out = out; p->args.out_dt = out_dtype;
  return run_steps(h, p, 0, p->steps.size(), s);
}

int avh_forward_ragged(avh_handle* h, const void* video, int video_dtype, const void* audio, int audio_dtype,
                       const int64_t* audio_strides, const int32_t* lengths, int B, int T, int output_layer, void* out,
                       int out_dtype, void* stream) {
  AVH_CHECK(h != nullptr, "null handle");
  AVH_CHECK(h->finalized, "weights not finalized (call avh_finalize_weights)");
  AVH_CHECK(h->cfg.compute_mode == AVH_COMPUTE_BF16, "packed ragged batches run in bf16 mode only (use avh_forward)");
  AVH_CHECK(h->cfg.reserved[0] == 0, "this handle holds a bare TransformerEncoder: use avh_encoder_forward");
  AVH_CHECK(video != nullptr || audio != nullptr, "both modalities are None");
  AVH_CHECK(lengths != nullptr && out != nullptr, "null argument");
  AVH_CHECK(B >= 1 && T >= 1 && B <= 4096, "bad batch");
  AVH_CHECK(output_layer >= 0 && output_layer <= h->cfg.encoder_layers, "output_layer out of range");
  AVH_CHECK(audio == nullptr || audio_strides != nullptr, "audio strides required");
  long long N = 0;
  int tmax = 0;
  for (int b = 0; b < B; ++b) {
    AVH_CHECK(lengths[b] >= 1 && lengths[b] <= T, "clip lengths must be in [1, T]");
    N += lengths[b];
    tmax = lengths[b] > tmax ? lengths[b] : tmax;
  }
  AVH_CHECK(N < (1ll << 24), "batch too large");
  AVH_CUDA_OK(cudaSetDevice(h->device));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (video != nullptr && video_dtype == AVH_U8) {
    avh_handle::Staging& st = h->staging[stream];
    if (avh::ensure_cap(&st.video_pp, &st.video_pp_cap, (size_t)B * T * 7744 * 2)) return 1;
    if (avh::launch_video_preprocess(reinterpret_cast<const unsigned char*>(video), (long long)B * T, h->vp_src_h,
                                     h->vp_src_w, 88, h->vp_mean, h->vp_std, st.video_pp, AVH_BF16, nullptr, s))
      return 1;
    video = st.video_pp;
    video_dtype = AVH_BF16;
  }
  AVH_CHECK(video == nullptr || video_dtype == AVH_F32 || video_dtype == AVH_F16 || video_dtype == AVH_BF16, "bad video dtype");
  // one plan per (clips, 128-row bucket of the packed rows, attention tiling class of the longest clip)
  const long long Nb = (N + 127) / 128 * 128;
  const int Tcap = tmax <= 160 ? 160 : (tmax + 127) / 128 * 128;
  avh::PlanKey key;
  key.kind = avh::PlanKind::Ragged;
  key.B = B; key.T = Tcap;
  key.has_video = video != nullptr; key.has_audio = audio != nullptr;
  key.output_layer = output_layer;
  key.ragged_rows = Nb;
  key.stream = s;
  avh::Plan* p = avh::get_plan(h, key);
  if (p == nullptr) return 1;
  h->last_plan = p;
  // per-call geometry -> pinned mirror -> device descriptor (ordered on the stream before the launches that read it)
  const int slot = p->rag_next;
  p->rag_next = (slot + 1) % avh::Plan::RAG_SLOTS;
  AVH_CUDA_OK(cudaEventSynchronize(p->rag_done[slot]));       // the copy that last used this mirror has run
  int* rh = p->rag_host[slot];
  rh[1] = (int)N;
  int acc = 0;
  for (int b = 0; b < B; ++b) { rh[16 + b] = acc; acc += lengths[b]; }
  rh[16 + B] = acc;
  int used_ints = 16 + B + 1;
  if (video != nullptr) {
    const int n_items = avh::stem_fused_ragged_items(lengths, B, avh::device_sm_count(),
                                                     reinterpret_cast<int4*>(rh + p->rag_items_off), p->rag_max_items);
    AVH_CHECK(n_items >= 0, "stem work list overflow");
    rh[0] = n_items;
    used_ints = p->rag_items_off + 4 * n_items;
  } else rh[0] = 0;
  AVH_CUDA_OK(cudaMemcpyAsync(p->rag, rh, (size_t)used_ints * 4, cudaMemcpyHostToDevice, s));
  AVH_CUDA_OK(cudaEventRecord(p->rag_done[slot], s));
  p->args.video = video; p->args.video_dt = video_dtype;
  p->args.audio = audio; p->args.audio_dt = audio_dtype;
  if (audio) for (int i = 0; i < 3; ++i) p->args.as[i] = audio_strides[i];
  p->args.mask = nullptr;
  p->args.out = out; p->args.out_dt = out_dtype;
  p->args.pitch = T;
  return run_steps(h, p, 0, p->steps.size(), s);
}

int avh_set_video_preprocess(avh_handle* h, int src_h, int src_w, double mean, double stdv) {
  AVH_CHECK(h != nullptr, "null handle");
  AVH_CHECK(src_h >= 88 && src_w >= 88 && src_h <= 4096 && src_w <= 4096, "raw frames must be at least 88 x 88");
  AVH_CHECK(stdv != 0.0, "std must be non-zero");
  h->vp_src_h = src_h; h->vp_src_w = src_w; h->vp_mean = mean; h->vp_std = stdv;
  return 0;
}

int avh_video_preprocess(const uint8_t* frames, int64_t n_frames, int src_h, int src_w, int crop, double mean,
                         double stdv, void* out, int out_dtype, void* stream) {
  AVH_CHECK(frames != nullptr && out != nullptr, "null argument");
  AVH_CHECK(out_dtype == AVH_F32 || out_dtype == AVH_F16 || out_dtype == AVH_BF16, "bad output dtype");
  return avh::launch_video_preprocess(frames, n_frames, src_h, src_w, crop, mean, stdv, out, out_dtype, nullptr,
                                      reinterpret_cast<cudaStream_t>(stream));
}

int avh_set_profiling(avh_handle* h, int on) {
  AVH_CHECK(h != nullptr, "null handle");
  h->profiling = on != 0;
  h->prof_plan = nullptr;
  return 0;
}

int avh_profile_json(avh_handle* h, char* buf, int64_t cap) {
  AVH_CHECK(h != nullptr && buf != nullptr && cap > 2, "bad argument");
  AVH_CHECK(h->prof_plan != nullptr, "no profiled forward recorded (avh_set_profiling(h,1) then avh_forward)");
  AVH_CUDA_OK(cudaSetDevice(h->device));
  avh::Plan* p = h->prof_plan;
  std::map<std::string, std::array<double, 3>> agg;     // name -> launches, ms, flops
  for (size_t i = 0; i < p->steps.size(); ++i) {
    AVH_CUDA_OK(cudaEventSynchronize(h->prof_events[2 * i + 1]));
    float ms = 0.f;
    AVH_CUDA_OK(cudaEventElapsedTime(&ms, h->prof_events[2 * i], h->prof_events[2 * i + 1]));
    auto& a = agg[p->steps[i].name];
    a[0] += 1; a[1] += ms; a[2] += p->steps[i].flops;
  }
  std::string out = "{";
  bool first = true;
  for (auto& kv : agg) {
    char tmp[256];
    snprintf(tmp, sizeof(tmp), "%s\"%s\": {\"launches\": %.0f, \"ms\": %.6f, \"tc_flops\": %.0f}", first ? "" : ", ",
             kv.first.c_str(), kv.second[0], kv.second[1], kv.second[2]);
    out += tmp;
    first = false;
  }
  out += "}";
  AVH_CHECK((int64_t)out.size() + 1 <= cap, "profile buffer too small");
  std::memcpy(buf, out.c_str(), out.size() + 1);
  return 0;
}

int avh_forward_host_async(avh_handle* h, const void* video, int video_dtype, const void* audio, int audio_dtype,
                           const uint8_t* padding_mask, int B, int T, int output_layer, void* out, int out_dtype,
                           void* stream) {
  AVH_CHECK(h != nullptr, "null handle");
  AVH_CUDA_OK(cudaSetDevice(h->device));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  avh_handle::Staging& st = h->staging[stream];
  const int D = h->cfg.encoder_embed_dim, Fa = h->cfg.audio_feat_dim;
  const size_t vbytes = video_dtype == AVH_U8 ? (size_t)B * T * h->vp_src_h * h->vp_src_w
                                              : (size_t)B * T * 88 * 88 * avh::dtype_size(video_dtype);
  const size_t abytes = (size_t)B * T * Fa * avh::dtype_size(audio_dtype);
  const size_t obytes = (size_t)B * T * D * avh::dtype_size(out_dtype);
  if (video) {
    if (avh::ensure_cap(&st.video, &st.video_cap, vbytes)) return 1;
    AVH_CUDA_OK(cudaMemcpyAsync(st.video, video, vbytes, cudaMemcpyHostToDevice, s));
  }
  if (audio) {
    if (avh::ensure_cap(&st.audio, &st.audio_cap, abytes)) return 1;
    AVH_CUDA_OK(cudaMemcpyAsync(st.audio, audio, abytes, cudaMemcpyHostToDevice, s));
  }
  if (padding_mask) {
    if (avh::ensure_cap(&st.mask, &st.mask_cap, (size_t)B * T)) return 1;
    AVH_CUDA_OK(cudaMemcpyAsync(st.mask, padding_mask, (size_t)B * T, cudaMemcpyHostToDevice, s));
  }
  if (avh::ensure_cap(&st.out, &st.out_cap, obytes)) return 1;
  const int64_t as[3] = {(int64_t)Fa * T, T, 1};
  if (avh_forward(h, video ? st.video : nullptr, video_dtype, audio ? st.audio : nullptr, audio_dtype, as,
                  padding_mask ? reinterpret_cast<const uint8_t*>(st.mask) : nullptr, B, T, output_layer, st.out,
                  out_dtype, stream))
    return 1;
  AVH_CUDA_OK(cudaMemcpyAsync(out, st.out, obytes, cudaMemcpyDeviceToHost, s));
  return 0;
}

int avh_forward_host(avh_handle* h, const void* video, int video_dtype, const void* audio, int audio_dtype,
                     const uint8_t* padding_mask, int B, int T, int output_layer, void* out, int out_dtype,
                     void* stream) {
  if (avh_forward_host_async(h, video, video_dtype, audio, audio_dtype, padding_mask, B, T, output_layer, out,
                             out_dtype, stream))
    return 1;
  AVH_CUDA_OK(cudaStreamSynchronize(reinterpret_cast<cudaStream_t>(stream)));
  return 0;
}

int avh_read_stage(avh_handle* h, const char* name, float* dst, int64_t capacity_elems, void* stream) {
  AVH_CHECK(h != nullptr && name != nullptr && dst != nullptr, "null argument");
  for (auto& kv : h->plans) {
    if (h->last_plan != nullptr && kv.second.get() != h->last_plan) continue;     // the most recent forward's plan
    auto it = kv.second->stages.find(name);
    if (it == kv.second->stages.end()) continue;
    const long long n = it->second.second.second;
    AVH_CHECK(n <= capacity_elems, "destination too small");
    return avh::launch_convert(it->second.first, it->second.second.first, dst, avh::DT_F32, n,
                               reinterpret_cast<cudaStream_t>(stream));
  }
  avh::set_last_error(std::string("no such stage in any cached plan: ") + name);
  return 1;
}

int avh_fbank(const int16_t* wav, const int64_t* offsets, const int32_t* video_len, int n_clips, int T,
              int normalize, float* out, uint8_t* padding_mask, void* stream) {
  avh::FbankArgs a;
  a.wav = wav;
  a.offsets = reinterpret_cast<const long long*>(offsets);
  a.video_len = video_len;
  a.n_clips = n_clips;
  a.T = T;
  a.normalize = normalize;
  a.out = out;
  a.padding_mask = padding_mask;
  return avh::launch_fbank(a, reinterpret_cast<cudaStream_t>(stream));
}

int avh_add_noise(const int16_t* wav, const int64_t* offsets, int n_clips, const float* noise, int64_t noise_len,
                  float snr_db, int16_t* out, double* scratch, void* stream) {
  return avh::launch_add_noise(wav, reinterpret_cast<const long long*>(offsets), n_clips, noise, noise_len, snr_db,
                               out, scratch, reinterpret_cast<cudaStream_t>(stream));
}

int avh_attention_bf16(const void* qkv, const uint8_t* padding_mask, const int32_t* cu_rows, int64_t rows, int B, int T,
                       int D, int H, int impl, void* out, void* stream) {
  AVH_CHECK(qkv != nullptr && out != nullptr, "null pointer");
  AVH_CHECK(impl == 0 || impl == 1, "impl must be 0 (mma.sync) or 1 (tcgen05)");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (impl == 0) {
    AVH_CHECK(cu_rows == nullptr, "the mma.sync kernel takes dense [B, T] batches only");
    return avh::launch_attention(qkv, padding_mask, out, B, T, D, H, 0, s);
  }
  avh::AttnTcPlan plan;
  if (avh::attention_tc_plan(qkv, rows, B, T, D, H, &plan)) return 1;
  return avh::attention_tc_launch(plan, padding_mask, cu_rows, out, s);
}

int avh_gemm_set_trace(void* dev_buf) {
  avh::gemm_set_trace(reinterpret_cast<unsigned long long*>(dev_buf));
  return 0;
}

int avh_gemm_bf16(const void* A, const void* B, int64_t M, int N, int K, const float* bias, int gelu, const void* R,
                  int r_fp32, void* C, int c_fp32, int block_n, int pair, int occ, void* stream) {
  AVH_CHECK(A && B && C, "null pointer");
  AVH_CHECK(K % 8 == 0 && N % 32 == 0, "K must be a multiple of 8 and N of 32");
  avh::GemmProblem pr;
  pr.A = A; pr.a_rows = M; pr.a_cols = K; pr.lda = K;
  pr.B = B; pr.b_rows = N; pr.b_cols = K; pr.ldb = K;
  pr.M = M; pr.N = N; pr.num_kb = (K + 63) / 64;
  // debug (tools/gemm_sweep.py): AVH_GEMM_KREPEAT=r walks the K range r times (L2-resident long main loops)
  static void* d_ktab = nullptr;
  const char* rep = std::getenv("AVH_GEMM_KREPEAT");
  if (rep != nullptr && std::atoi(rep) > 1) {
    const int r = std::atoi(rep), kb0 = pr.num_kb;
    AVH_CHECK(kb0 * r <= avh::GEMM_MAX_KSTEPS, "k repeat too large");
    std::vector<avh::KStep> t;
    for (int i = 0; i < kb0 * r; ++i) t.push_back(avh::KStep{(i % kb0) * 64, 0, (i % kb0) * 64, 0});
    if (d_ktab == nullptr) AVH_CUDA_OK(cudaMalloc(&d_ktab, avh::GEMM_MAX_KSTEPS * sizeof(avh::KStep)));
    AVH_CUDA_OK(cudaMemcpy(d_ktab, t.data(), t.size() * sizeof(avh::KStep), cudaMemcpyHostToDevice));
    pr.ktable = reinterpret_cast<const avh::KStep*>(d_ktab);
    pr.num_kb = kb0 * r;
  }
  pr.block_n = block_n;
  pr.pair = pair;
  pr.occ = occ;
  {   // stream-K workspace for the stand-alone entry point (tests, tools): one per device, allocated on first use
    static std::map<int, std::pair<float*, int*>> ws;
    int dev = 0;
    AVH_CUDA_OK(cudaGetDevice(&dev));
    const size_t bytes = (size_t)avh::device_sm_count() * 128 * 256 * 4;
    if (ws.find(dev) == ws.end()) {
      float* w = nullptr; int* f = nullptr;
      AVH_CUDA_OK(cudaMalloc(&w, bytes));
      AVH_CUDA_OK(cudaMalloc(&f, 4096));
      AVH_CUDA_OK(cudaMemset(f, 0, 4096));
      ws[dev] = {w, f};
    }
    pr.sk_ws = ws[dev].first; pr.sk_ws_bytes = bytes; pr.sk_flags = ws[dev].second;
  }
  pr.ep.C = C; pr.ep.ldc = N; pr.ep.c_fp32 = c_fp32;
  pr.ep.col_bias = bias;
  pr.ep.act = gelu ? avh::ACT_GELU : avh::ACT_NONE;
  pr.ep.R = R; pr.ep.ldr = N; pr.ep.r_fp32 = r_fp32;
  avh::GemmPlan plan;
  if (avh::gemm_plan(pr, &plan)) return 1;
  return avh::gemm_launch(plan, reinterpret_cast<cudaStream_t>(stream));
}

}  // extern "C"
