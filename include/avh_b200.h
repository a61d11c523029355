/* avh_b200.h — C ABI of libavh_b200.so: the sm_100a (B200) implementation of the AV-HuBERT encoder hot path.
 *
 * The reference (EnriqueOO97/MultiModalVC) is pure Python/PyTorch and has no FFI of its own; the entry
 * points below are what a binding for this path replaces, call for call:
 *
 *   avh_create / avh_load_tensor / avh_finalize_weights
 *       <- AVHubertModel.__init__ + nn.Module.load_state_dict(state["model"], strict=False)
 *          (avhubert/hubert.py:335-433, src/model.py:218-226, avhubert/hubert_asr.py:299-305)
 *   avh_forward
 *       <- AVHubertModel.extract_finetune(source={'audio','video'}, padding_mask, output_layer)
 *          (avhubert/hubert.py:694-745) including ResEncoder.forward (avhubert/resnet.py:156-164) and
 *          TransformerEncoder.forward (fairseq/fairseq/models/wav2vec/wav2vec2.py:859-902)
 *   avh_forward_host
 *       <- the same call preceded by utils.move_to_cuda(sample) (src/eval.py:196) and followed by a
 *          device->host read of the features: the end-to-end path with HOST buffers
 *   avh_fbank
 *       <- logfbank + stacker + audio/video length alignment + per-frame F.layer_norm + collater_audio
 *          (avhubert/hubert_dataset.py:286-296,351-353,430-456)
 *   avh_add_noise
 *       <- AVHubertDataset.add_noise with the noise clip already selected (avhubert/hubert_dataset.py:317-346)
 *   avh_video_preprocess, and avh_forward* with video_dtype == AVH_U8 (+ avh_set_video_preprocess)
 *       <- AVHubertDataset.load_video's eval transform: Normalize(0,255) -> CenterCrop(88) -> Normalize(mean,std)
 *          (avhubert/hubert_dataset.py:222-226,298-302; avhubert/utils.py:56-95), i.e. raw uint8 gray frames go
 *          host->device (4x fewer bytes than fp32) and are normalised on the device (SURVEY 8(f)-1)
 *
 * Conventions: every function returns 0 on success and non-zero on failure; avh_last_error() returns the
 * message of the last failure on the calling thread.  No exceptions cross the boundary.  All work is
 * enqueued on the CUDA stream passed in (a cudaStream_t cast to void*; NULL = legacy default stream) with no
 * device-wide synchronisation.  The caller owns every input/output buffer; the library only borrows the
 * pointers for the duration of the enqueue and never writes to inputs.  A handle is bound to one device
 * and is not thread-safe; use one handle per device/thread (one process per GPU in the reference:
 * fairseq/fairseq/distributed/utils.py:317-350).
 */
#ifndef AVH_B200_H_
#define AVH_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AVH_ABI_VERSION 1
#if defined(__GNUC__)
#define AVH_API __attribute__((visibility("default")))
#else
#define AVH_API
#endif

/* element types of caller-provided buffers */
enum { AVH_F32 = 0, AVH_F16 = 1, AVH_BF16 = 2, AVH_U8 = 3 /* raw video frames only */ };
/* arithmetic of the dense contractions */
enum {
  AVH_COMPUTE_BF16 = 0, /* bf16 operands, fp32 accumulation (tcgen05 kind::f16) */
  AVH_COMPUTE_FP32 = 1  /* fp32-faithful: operands split into bf16 hi+mid planes, 3 tcgen05 products, fp32 accumulation */
};
enum { AVH_FUSE_CONCAT = 0, AVH_FUSE_ADD = 1 };

/* Mirror of the AVHubertConfig fields that determine shapes on this path (avhubert/hubert.py:64-315). */
typedef struct avh_config {
  int32_t encoder_layers;          /* hubert.py:76  */
  int32_t encoder_embed_dim;       /* hubert.py:79  */
  int32_t encoder_ffn_embed_dim;   /* hubert.py:82  */
  int32_t encoder_attention_heads; /* hubert.py:85  (head dim must be 64) */
  int32_t audio_feat_dim;          /* hubert.py:236 (104 = 4 x 26 stacked log-fbank) */
  int32_t modality_fuse;           /* hubert.py:238 AVH_FUSE_* */
  int32_t layer_norm_first;        /* hubert.py:131 */
  int32_t conv_pos;                /* hubert.py:213 (128) */
  int32_t conv_pos_groups;         /* hubert.py:217 (16)  */
  int32_t compute_mode;            /* AVH_COMPUTE_* */
  int32_t frontend_chunk_frames;   /* video frames per lip-frontend pass; 0 = default.  avh_forward_train runs the whole
                                      batch in one pass (BatchNorm batch statistics) */
  int32_t capture_stages;          /* non-zero: keep copies of intermediate stages for avh_read_stage (tests) */
  int32_t reserved[4];             /* reserved[0] = 1: the handle holds a bare fairseq TransformerEncoder (state-dict keys
                                      "encoder.*" only; avh_encoder_forward is its one forward entry point);
                                      reserved[0] = 2: a Q-Former (avh_qformer_forward; reserved[1] = encoder_width,
                                      reserved[2] = rows of query_tokens);
                                      reserved[3] = 1: trainable encoder (also packs the transposed weights the
                                      backward needs: avh_encoder_train_forward / avh_encoder_backward) */
} avh_config;

typedef struct avh_handle avh_handle;

AVH_API int avh_abi_version(void);
AVH_API const char* avh_last_error(void);

AVH_API int avh_create(const avh_config* cfg, int device, avh_handle** out);
AVH_API int avh_destroy(avh_handle* h);

/* One state-dict entry, by its reference key name (e.g. "encoder.layers.3.fc1.weight",
 * "feature_extractor_video.resnet.trunk.layer2.0.downsample.1.running_var").  `data` may be a host or a
 * device pointer (contiguous, `dtype` elements).  Keys the path never reads (mask_emb, final_proj.*,
 * label_embs_concat, *.num_batches_tracked) are accepted and ignored.  Unknown keys fail. */
AVH_API int avh_load_tensor(avh_handle* h, const char* key, const void* data, int dtype, const int64_t* shape, int ndim);
/* Fold eval-mode BatchNorm into conv epilogues, fold weight-norm of pos_conv, fold the q scaling, repack
 * every weight into the kernels' K-major bf16 layouts and upload.  Fails listing the first missing key. */
AVH_API int avh_finalize_weights(avh_handle* h);
/* Frees the fp32 host copies avh_load_tensor keeps for re-finalisation (~1.3 GB for Large).  After this call a
 * weight update must re-load EVERY tensor before the next avh_finalize_weights (nn.Module.load_state_dict does). */
AVH_API int avh_drop_host_weights(avh_handle* h);
/* Drains `stream`, then frees the execution plans, workspaces and host-path staging buffers bound to it (a caller
 * retiring a CUDA stream; torch.cuda.Stream objects going out of scope). */
AVH_API int avh_release_stream(avh_handle* h, void* stream);

/* extract_finetune.  All pointers are DEVICE pointers.
 *   video  [B,1,T,88,88] contiguous (AVH_F32/F16/BF16), or raw [B,1,T,src_h,src_w] uint8 frames (AVH_U8, see
 *          avh_set_video_preprocess), or NULL (zero-filled modality arm, hubert.py:703-704)
 *   audio  [B,F,T] with element strides audio_strides[3] (the collater hands a transposed view,
 *          hubert_dataset.py:453), or NULL (hubert.py:705-708)
 *   padding_mask [B,T] bytes, non-zero = padded frame, or NULL
 *   output_layer 0 = all layers + final LayerNorm; k>=1 = stop after layer k, no final LayerNorm
 *          (hubert.py:742, wav2vec2.py:862,892-894)
 *   out    [B,T,D] contiguous, out_dtype elements */
AVH_API int avh_forward(avh_handle* h, const void* video, int video_dtype, const void* audio, int audio_dtype,
                const int64_t* audio_strides, const uint8_t* padding_mask, int B, int T, int output_layer,
                void* out, int out_dtype, void* stream);

/* extract_finetune with the module in TRAINING mode and no gradient — what MMS-LLaMA's frozen encoder executes during
 * training (src/model.py:96-100,280: requires_grad False + no_grad, but the module follows model.train()):
 *   BatchNorm2d/3d normalise with BATCH statistics and update running_mean / running_var (avhubert/resnet.py:23,44,56,139);
 *   nn.Dropout at hubert.py:729 (dropout_input), wav2vec2.py:879 (dropout), :980,:990 (dropout1 / dropout3 = dropout),
 *   :987 (dropout2 = activation_dropout) — Philox masks of this library's own stream (seed per call);
 *   LayerDrop (wav2vec2.py:887-888): the caller draws the coins and passes layer_skip (HOST, one byte per layer).
 * GradMultiply (fairseq/fairseq/modules/grad_multiply.py) is the identity in a forward.  attention_dropout must be 0.
 * Same tensors as avh_forward (float video only).  The updated running statistics are read with avh_read_bn_stats:
 * flat fp32, per BatchNorm (running_mean[C], running_var[C]) in the order frontend3D.1, then for layer1..4, block 0..1:
 * bn1, bn2, downsample.1 (when present).  Eval-mode forwards keep using the statistics folded at the last
 * avh_finalize_weights until the caller re-folds them (avh_refresh_eval_weights_device) or re-loads them. */
typedef struct avh_train_args {
  float dropout_input, dropout, activation_dropout, attention_dropout;
  float bn_momentum;               /* nn.BatchNorm default 0.1 */
  uint64_t seed;                   /* dropout stream of this call */
  const uint8_t* layer_skip;       /* HOST [encoder_layers], non-zero = layer dropped; NULL = keep all */
} avh_train_args;
AVH_API int avh_forward_train(avh_handle* h, const void* video, int video_dtype, const void* audio, int audio_dtype,
                              const int64_t* audio_strides, const uint8_t* padding_mask, int B, int T, int output_layer,
                              const avh_train_args* args, void* out, int out_dtype, void* stream);
/* First consumer of the encoder output in MMS-LLaMA (SURVEY 8(f)-3, src/model.py:596-609): the per-sample loop
 * F.interpolate(av_feat[b][:len_in[b]].T[None], size=len_out[b], mode='linear').T into a zero-padded batch + mask, as
 * one launch.  x [B,T,C], len_in / len_out int32 [B] (DEVICE), out [B,Tout,C] (same dtype, rows >= len_out[b] zero),
 * mask int64 [B,Tout] (1 = valid) or NULL.  Index arithmetic of ATen's upsample_linear1d (align_corners=False). */
AVH_API int avh_interp_linear(const void* x, int dtype, int B, int T, int C, const int32_t* len_in, const int32_t* len_out,
                              int Tout, void* out, int64_t* mask, void* stream);

/* Pretraining-mode extras (SURVEY 8(f)-4).
 * avh_mask_substitute = the tensor side of AVHubertModel.apply_input_mask (avhubert/hubert.py:442-494) and
 * apply_feature_mask (:496-536): the host draws the spans (compute_mask_indices, avhubert/utils.py:142-270) and gives ONE
 * int32 code per (clip, frame) [B*T] (device): >= 0 take frame b'*T+t' of x, -1 keep, -2 zeros, -3 the mask embedding
 * `emb` [U] (device).  Out of place; every source is read from the un-substituted x, as the reference's right-hand
 * side is.  layout 0: contiguous units x = [B,T,U] (video [B,1,T,88*88], token rows [B,T,C]); channel_zero [B,U] bytes
 * (may be NULL) zeroes channels of every frame of a clip (mask_channel_prob).  layout 1: x = [B,U,T] with element
 * `strides` (the collater's transposed audio view), out contiguous [B,U,T]. */
AVH_API int avh_mask_substitute(const void* x, int dtype, int layout, const int64_t* strides, int B, int T, int U,
                                const int32_t* code, const void* emb, int emb_dtype, const uint8_t* channel_zero,
                                void* out, int out_dtype, void* stream);
/* AVHubertModel.compute_logits (avhubert/hubert.py:576-589): out[m,v] = (<feats_m, emb_v> + bias[v]) / logit_temp for
 * sim_type 0 ('dot'), divided by max(|feats_m| |emb_v|, 1e-6) first for sim_type 1 ('cosine'); fp32 arithmetic.
 * feats [M,K] (row stride ldf), emb [V,K] (row stride lde), bias fp32 [V] or NULL, out fp32 [M,V] (row stride ldo).
 * With sim_type 0, logit_temp 1 and a bias this is final_proj (nn.Linear, hubert.py:654). */
AVH_API int avh_compute_logits(const void* feats, int f_dtype, int64_t ldf, const void* emb, int e_dtype, int64_t lde,
                               const float* bias, int64_t M, int V, int K, int sim_type, float logit_temp, float* out,
                               int64_t ldo, void* stream);
/* *acc (device double) = sum of x[i]^2 — features_pen = features.float().pow(2).mean() (hubert.py:629) times numel. */
AVH_API int avh_sum_squares(const void* x, int dtype, int64_t n, double* acc, void* stream);
/* Backward of avh_compute_logits, same argument conventions: from the forward's feats, emb, logits (fp32 [M,V], read by
 * sim_type 1 only; may be NULL for 'dot') and dlogits = dL/dlogits (fp32 [M,V]; logits and dlogits share the row stride
 * ldo), writes dfeats = dL/dfeats (fp32 [M,K], row stride ldd_f), demb = dL/demb (fp32 [V,K], row stride ldd_e) and
 * dbias = dL/dbias (fp32 [V]); any of the three may be NULL.  Cosine: where |feats_m| |emb_v| < 1e-6 the clamped
 * denominator is a constant (torch.clamp's gradient).  fp32 arithmetic, every reduction in a fixed order (repeat calls are
 * bit-identical).  With sim_type 0, logit_temp 1 this is the backward of final_proj. */
AVH_API int avh_compute_logits_backward(const void* feats, int f_dtype, int64_t ldf, const void* emb, int e_dtype, int64_t lde,
                                        int64_t M, int V, int K, int sim_type, float logit_temp, const float* logits,
                                        const float* dlogits, int64_t ldo, float* dfeats, int64_t ldd_f, float* demb,
                                        int64_t ldd_e, float* dbias, void* stream);

/* Kernel-level entry point of the dropout used above (tests): x[i] = keep(i) ? x[i] / (1 - p) : 0 in place, keep(i) a
 * pure function of (seed, site, i) through Philox4x32-10 — nn.Dropout semantics, this library's own random stream. */
AVH_API int avh_dropout(void* x, int dtype, int64_t n, float p, uint64_t seed, uint32_t site, void* stream);
AVH_API int avh_bn_stats_count(avh_handle* h, int64_t* n_floats);
AVH_API int avh_read_bn_stats(avh_handle* h, float* dst, int64_t capacity, void* stream);

/* fairseq TransformerEncoder.forward(x, padding_mask, layer) (fairseq/fairseq/models/wav2vec/wav2vec2.py:859-902) on
 * caller-provided features x [B,T,D] (device, AVH_F32/F16/BF16): padded frames zeroed, positional conv + GELU, the
 * layers, final LayerNorm when pre-LN and output_layer == 0; out [B,T,D].  Works on any finalised handle (it uses the
 * "encoder.*" weights); a handle created with reserved[0] != 0 needs no other weights — the encoder of
 * src/sub_model/modules.py:108-142 (Speech_Rate_Predictor, d = 256) is served this way. */
AVH_API int avh_encoder_forward(avh_handle* h, const void* x, int x_dtype, const uint8_t* padding_mask, int B, int T,
                                int output_layer, void* out, int out_dtype, void* stream);

/* Training step of the TransformerEncoder (SURVEY 8(a) row A18, encoder part of BASELINE config 5; pre-LN or post-LN
 * layers as layer_norm_first says): forward with saved activations, then the backward of exactly that graph —
 * wav2vec2.py:859-902 (positional conv + GELU + residual, index_put on padded frames), :974-992 (pre-LN layer) or
 * :993-1012 (post-LN layer), multihead_attention.py:170-192, the final LayerNorm (:862-863, pre-LN) or the LayerNorm after
 * the positional conv (:876-877, post-LN) — what torch.autograd computes for the reference module.  Dropout and LayerDrop as avh_set_train_args
 * leaves them for the call (none without it).
 * Handle: any handle with encoder weights created with avh_config.reserved[3] = 1 (packs W^T for the dX = dY W GEMMs).
 * avh_encoder_train_forward: as avh_encoder_forward (all layers, + final LayerNorm when pre-LN); avh_encoder_backward:
 * dout [B,T,D] = dL/d(out) (every row counts, padded frames too, as under autograd), dx [B,T,D] = dL/d(x) (may be NULL), grads = fp32 [avh_encoder_grad_count]
 * (may be NULL) in this order: per layer {q,k,v}_proj.weight, {q,k,v}_proj.bias, out_proj.weight, out_proj.bias,
 * self_attn_layer_norm.{weight,bias}, fc1.weight, fc1.bias, fc2.weight, fc2.bias, final_layer_norm.{weight,bias}; then
 * encoder.layer_norm.{weight,bias}; then pos_conv.0.{bias, weight_g, weight_v}.  Same stream as the forward. */
AVH_API int avh_encoder_grad_count(avh_handle* h, int64_t* n_floats);
AVH_API int avh_encoder_train_forward(avh_handle* h, const void* x, int x_dtype, const uint8_t* padding_mask, int B, int T,
                                      void* out, int out_dtype, void* stream);
AVH_API int avh_encoder_backward(avh_handle* h, const void* dout, int dout_dtype, void* dx, int dx_dtype, float* grads,
                                 int64_t grads_capacity, void* stream);
/* The same backward with the gradients handed over BUCKET BY BUCKET, so that the gradient all-reduce of the training
 * configuration (fairseq legacy_distributed_data_parallel.py:76-165, SURVEY row A19) overlaps the rest of the backward:
 * the flat buffer is cut into buckets in the order the backward completes them (four encoder layers each, last layers
 * first; then final LayerNorm + positional conv + fusion tail; then the feature extractors).  As soon as a bucket is
 * final it is converted into `grads` (fp32 / bf16 / fp16 [avh_encoder_grad_count], same element offsets) and an event is
 * recorded; avh_grad_bucket_wait makes another stream wait for bucket k of the last avh_encoder_backward_buckets call
 * (the caller then issues its collective there).  Bucket geometry is a property of the last training forward's plan. */
AVH_API int avh_encoder_backward_buckets(avh_handle* h, const void* dout, int dout_dtype, void* dx, int dx_dtype, void* grads,
                                         int grads_dtype, int64_t grads_capacity, void* stream);
AVH_API int avh_grad_bucket_count(avh_handle* h, int32_t* count);
/* After an optimizer step on a trainable handle (avh_config.reserved[3] = 1): rewrite, IN PLACE and on the device, every
 * packed tensor the TRAINING plans read (K-major bf16 planes of every Linear / convolution and their transposes, biases,
 * LayerNorm / BatchNorm affine parameters, PReLU slopes, the weight-normed positional convolution) from the caller's
 * device-resident parameters: names[i] = state-dict key (the reference's names, as avh_load_tensor), ptrs[i] = device
 * pointer of the contiguous tensor, dtypes[i] = AVH_F32 / AVH_F16 / AVH_BF16, numels[i] = element count.  Plans and
 * captured graphs stay valid (no pointer moves); nothing crosses the host (avh_finalize_weights re-packs through the
 * host: seconds for the Large model).  The eval-only packed forms (BatchNorm folded with the running statistics, the
 * conv2 + shortcut GEMM weights with both BatchNorm scales folded in) are NOT refreshed: before the next eval-mode
 * forward call avh_refresh_eval_weights_device.  Enqueued on `stream`. */
AVH_API int avh_refresh_weights_device(avh_handle* h, const char* const* names, const void* const* ptrs, const int32_t* dtypes,
                                       const int64_t* numels, int32_t count, void* stream);
/* Before an eval-mode forward that follows training on the handle (optimizer steps, or training-mode forwards that moved
 * the BatchNorm running statistics): on a trainable handle the work of avh_refresh_weights_device, then on every
 * AV-HuBERT handle the eval-only forms — per BatchNorm scale = gamma / sqrt(running_var + 1e-5) and bias = beta -
 * running_mean * scale, the fp32 gamma / beta / running statistics the training-mode BatchNorm starts from, and the conv2
 * + shortcut GEMM weights of layers 2-4 — in place, on the device, bit-identical to what avh_finalize_weights computes
 * from the same values.  The list holds the parameters AND the BatchNorm buffers ("...running_mean",
 * "...running_var"), same arguments as avh_refresh_weights_device; plans, arenas and captured graphs stay valid.  The
 * job list is replayed as its own CUDA graph for the pointer set it was last called with.  Not for Q-Former handles. */
AVH_API int avh_refresh_eval_weights_device(avh_handle* h, const char* const* names, const void* const* ptrs,
                                            const int32_t* dtypes, const int64_t* numels, int32_t count, void* stream);
/* Number of execution plans the handle holds (forward and training plans, all streams); avh_finalize_weights drops them. */
AVH_API int avh_plan_count(avh_handle* h, int32_t* count);
AVH_API int avh_grad_bucket_range(avh_handle* h, int k, int64_t* begin, int64_t* end);       /* [begin, end) elements */
AVH_API int avh_grad_bucket_wait(avh_handle* h, int k, void* stream);

/* Regularisation of the NEXT avh_encoder_train_forward / avh_tail_train_forward / avh_full_train_forward on the handle,
 * which consumes it (without this call a training step has no dropout and drops no layer).  Same masks and sites as
 * avh_forward_train: dropout_input on the post_extract_proj output (tail and full steps only; ignored by the bare
 * encoder), dropout after the positional conv block and on the attention / FFN block outputs, activation_dropout after
 * the FFN GELU — element i of a site's [B*T, C] tensor keeps lane i % 4 of Philox4x32-10(seed, i / 4, site), exactly as
 * avh_dropout.  layer_skip (HOST [encoder_layers], or NULL = no LayerDrop) holds the LayerDrop coins: a dropped layer is
 * the identity, dx passes through it, and its 16 gradient tensors are zero in the flat buffer.  The backward
 * (avh_encoder_backward*) uses the seed and coins of its forward and regenerates the masks.  Probabilities select the
 * launch plan (and so its CUDA graphs), the seed and coins do not: a step replays its graphs for any seed and any set of
 * dropped layers.  attention_dropout must be 0; bn_momentum is not read (avh_full_train_forward takes its own). */
AVH_API int avh_set_train_args(avh_handle* h, const avh_train_args* args);

/* The trainable tail of AVHubertModel.extract_finetune when the feature extractors are frozen (feature_grad_mult <= 0: the
 * reference runs them under no_grad, avhubert/hubert.py:538-547): fused [B,T,E] = the concatenated / summed extractor
 * outputs BEFORE the fusion LayerNorm (avh_read_stage "fused"), then layer_norm -> post_extract_proj -> index_put ->
 * encoder (hubert.py:719-745) with saved activations; avh_encoder_backward then returns, after the encoder's gradients
 * in the order above, post_extract_proj.{weight,bias} (concat fusion only) and layer_norm.{weight,bias}; its dx is the
 * gradient at the ENCODER input (post_extract_proj output).  AV-HuBERT handle created with reserved[3] = 1. */
AVH_API int avh_tail_grad_count(avh_handle* h, int64_t* n_floats);
AVH_API int avh_tail_train_forward(avh_handle* h, const void* fused, int dtype, const uint8_t* padding_mask, int B, int T,
                                   void* out, int out_dtype, void* stream);      /* regularisation: avh_set_train_args */

/* The whole fine-tuning step (feature_grad_mult > 0, BASELINE config 5; dropout / LayerDrop: avh_set_train_args): lip
 * ResNet (training-mode BatchNorm:
 * batch statistics, running statistics updated with bn_momentum — read them back with avh_read_bn_stats), modality
 * projections, fusion, encoder, with saved activations; avh_encoder_backward then also returns, after the tail's
 * gradients, those of the feature extractors (scaled by feature_grad_mult as fairseq's GradMultiply does,
 * avhubert/hubert.py:538-547): feature_extractor_audio.proj.{weight [D, round_up(F,64)], bias} (when audio is given),
 * feature_extractor_video.proj.{weight, bias}, frontend3D.0.weight as [64, 5, 8, 8] (dt, kh, kw; kh = 7 / kw = 7 zero),
 * frontend3D.1.{weight,bias}, frontend3D.2.weight, and per BasicBlock conv1.weight as [C, kh, kw, Cin], bn1.{weight,
 * bias}, relu1.weight, conv2.weight, bn2.{weight,bias}, relu2.weight, downsample.0.weight [C, Cin], downsample.1.{weight,
 * bias} (first block of layers 2-4).  Every convolution of this path is explicit patches -> one GEMM (dense NHWC maps).
 * video [B,1,T,88,88] float (or NULL), audio [B,F,T] + strides (or NULL).  Its dx output is not defined (pass NULL). */
AVH_API int avh_full_grad_count(avh_handle* h, int has_video, int has_audio, int64_t* n_floats);
AVH_API int avh_full_train_forward(avh_handle* h, const void* video, int video_dtype, const void* audio, int audio_dtype,
                                   const int64_t* audio_strides, const uint8_t* padding_mask, int B, int T,
                                   float feature_grad_mult, float bn_momentum, void* out, int out_dtype, void* stream);

/* Pretraining step (AVHubertModel.forward in training mode, avhubert/hubert.py:591-674).  avh_set_modality_drop marks the
 * NEXT avh_forward_train or avh_full_train_forward on the handle, which consumes it, as a pretraining step that drops
 * `which` modality (0 none, 1 audio, 2 video: the reference's two coins, hubert.py:611-616, drawn by the caller).  Both
 * modalities must be given.  The dropped arm's projection output is zeros in the fused features, concat or add fusion;
 * the lip ResNet still runs when video is dropped (its BatchNorm running statistics move).  The backward of a full step
 * skips the dropped arm and writes zeros into its gradients.  The decision does not select the launch plan (a step
 * replays its CUDA graphs for any decision); marking a step does.  The frozen-extractor step (avh_tail_train_forward)
 * takes fused features that already hold the zeros.
 * avh_train_features_pen: *acc (device double) = sum of squares of the fused features [B,T,E] of the last training
 * forward on the handle (avh_forward_train, avh_tail_train_forward, avh_full_train_forward); features_pen = *acc / (B T E).
 * avh_set_features_pen_grad: after a marked avh_full_train_forward and before its backward, dL/dfeatures_pen (a device
 * float, NULL = 0; 0 unless set) — copied into the plan on `stream`; the backward adds (2 dL/dpen / (B T E)) fused to
 * dL/dfused before the feature_grad_mult scaling. */
AVH_API int avh_set_modality_drop(avh_handle* h, int which);
AVH_API int avh_train_features_pen(avh_handle* h, double* acc, void* stream);
AVH_API int avh_set_features_pen_grad(avh_handle* h, const float* dpen, void* stream);

/* The Q-Former that compresses the fused AV features into query tokens in MMS-LLaMA (SURVEY 8(f) rank 3):
 * Qformer.bert(query_embeds=query_tokens[:, :Lq], attention_mask, encoder_hidden_states=enc, encoder_attention_mask)
 * ['last_hidden_state'] (src/model.py:584-619 -> src/sub_model/Qformer.py:805-968, query-only path: self-attention over
 * the queries, cross-attention to enc, *_query feed-forward, post-LN, eps 1e-12, erf GELU).
 * Handle: avh_create with reserved[0] = 2, encoder_layers = qformer_layers, encoder_embed_dim = hidden size (heads x 64),
 * encoder_ffn_embed_dim = intermediate size, reserved[1] = encoder_width (features of enc), reserved[2] = rows of
 * query_tokens; avh_load_tensor with the BertModel-level state-dict keys ("embeddings.LayerNorm.*",
 * "encoder.layer.{i}.attention.self.{query,key,value}.*", ".attention.output.{dense,LayerNorm}.*", ".crossattention.*",
 * ".intermediate_query.dense.*", ".output_query.{dense,LayerNorm}.*") plus "query_tokens" [1, max_queries, hidden].
 * enc [B,Lk,encoder_width] (device, any float dtype); enc_padding [B,Lk] bytes, 1 = padded frame (the reference passes
 * the complement as a 0/1 long mask), or NULL; len_queries HOST int32 [B] valid queries per clip (rows beyond are masked
 * as keys of the self-attention, as query_attn_mask does) or NULL; out [B,Lq,hidden].  Masked keys are dropped — the
 * reference adds -10000 to their scores, which fp32 exp() turns into exactly 0 as long as one key is valid. */
AVH_API int avh_qformer_forward(avh_handle* h, const void* enc, int enc_dtype, const uint8_t* enc_padding,
                                const int32_t* len_queries, int B, int Lq, int Lk, void* out, int out_dtype, void* stream);

/* extract_finetune for RAGGED batches without computing on pad frames (SURVEY 7 step 9; BASELINE config 3): same
 * padded tensors as avh_forward (video [B,1,T,88,88] or raw uint8, audio [B,F,T] + strides, out [B,T,D]) plus the HOST
 * array lengths[B] (valid frames per clip, 1..T; padding must be a suffix, as the collater writes it,
 * hubert_dataset.py:433-447).  Inside, frames and tokens are packed back to back (sum(lengths) rows rounded up to
 * 128), attention runs per clip, and the output rows of pad positions are written as ZEROS — the one deviation from
 * the dense path, where the reference leaves non-zero values nobody reads behind the padding mask.  Valid positions
 * carry the same values as avh_forward with the equivalent padding mask (bf16 mode only). */
AVH_API int avh_forward_ragged(avh_handle* h, const void* video, int video_dtype, const void* audio, int audio_dtype,
                               const int64_t* audio_strides, const int32_t* lengths, int B, int T, int output_layer,
                               void* out, int out_dtype, void* stream);

/* Raw-video geometry for video_dtype == AVH_U8: video is then [B,1,T,src_h,src_w] uint8 gray frames (mouth ROI as
 * stored by the dataset, e.g. 96 x 96); avh_forward* first applies x/255, the centre crop to 88 x 88 with offsets
 * (src-88)/2 and (x-mean)/std (defaults 0.421 / 0.165, hubert_pretraining.py:144-149).  Default: 88 x 88 (no crop).
 * Frames flagged in padding_mask become 0.0 (the collater zero-pads AFTER the per-sample Normalize,
 * hubert_dataset.py:430-456), whatever bytes the caller left in them. */
AVH_API int avh_set_video_preprocess(avh_handle* h, int src_h, int src_w, double mean, double std);

/* The same transform as a stand-alone device op: frames [n_frames, src_h, src_w] uint8 -> out [n_frames, crop, crop]
 * (out_dtype AVH_F32 results are bit-identical to the reference's float64 numpy + cast).  crop % 8 == 0. */
AVH_API int avh_video_preprocess(const uint8_t* frames, int64_t n_frames, int src_h, int src_w, int crop, double mean,
                         double std, void* out, int out_dtype, void* stream);

/* Same computation with HOST buffers (pinned memory recommended): copies the inputs host->device, runs
 * avh_forward and copies `out` device->host, all on `stream`; returns after the stream has drained.
 * `audio` here is contiguous [B,F,T]. */
AVH_API int avh_forward_host(avh_handle* h, const void* video, int video_dtype, const void* audio, int audio_dtype,
                     const uint8_t* padding_mask, int B, int T, int output_layer, void* out, int out_dtype,
                     void* stream);

/* avh_forward_host without the final wait: everything is enqueued on `stream` (H2D, kernels, D2H) and the call
 * returns; `out` and the input buffers must stay valid until the caller has synchronised the stream.  Work
 * enqueued on different streams uses separate workspaces, so several batches can be in flight per device. */
AVH_API int avh_forward_host_async(avh_handle* h, const void* video, int video_dtype, const void* audio, int audio_dtype,
                           const uint8_t* padding_mask, int B, int T, int output_layer, void* out, int out_dtype,
                           void* stream);

/* Intermediate taps for stage-level parity tests; names: "resnet" [B*T,512], "fused" [B*T,E] (before the LayerNorm), "fused_ln" [B*T,E],
 * "enc_in" [B*T,D], and the lip-frontend maps "stem", "layer{L}.{b}.mid" / "layer{L}.{b}.out" (L = 1..4, b = 0, 1) and
 * "layer{L}.0.ds" (L = 2..4, fp32 mode and training mode only) — layouts in AVHubertModel.read_stage.  Copies the fp32
 * value of the last avh_forward into `dst` (device, fp32). */
AVH_API int avh_read_stage(avh_handle* h, const char* name, float* dst, int64_t capacity_elems, void* stream);

/* Audio frontend.  wav: int16 samples of n_clips clips back to back, clip i = [offsets[i], offsets[i+1]).
 *   video_len[i] (may be NULL): number of video frames clip i is aligned to (pad with zero rows / trim).
 *   T: collated length; rows >= the clip's own length are zero and flagged in padding_mask.
 *   out [n_clips, T, 104] fp32 row-major (the collater's [B,104,T] is the transposed VIEW of this),
 *   padding_mask [n_clips, T] bytes (may be NULL).  All DEVICE pointers. */
AVH_API int avh_fbank(const int16_t* wav, const int64_t* offsets, const int32_t* video_len, int n_clips, int T,
              int normalize, float* out, uint8_t* padding_mask, void* stream);

/* noise: fp32 noise clip (device) tiled/cropped to each clip's length from its start; snr_db as in the
 * reference; out int16 (device) same layout as wav; scratch: device buffer of >= 4*n_clips doubles. */
AVH_API int avh_add_noise(const int16_t* wav, const int64_t* offsets, int n_clips, const float* noise, int64_t noise_len,
                  float snr_db, int16_t* out, double* scratch, void* stream);

/* Kernel-level entry point of the attention core (tests, tools): qkv bf16 [rows, 3*D] = fused projection with q
 * pre-scaled by head_dim^-0.5, out bf16 [rows, D].  Dense batches: rows = B*T, clip b at row b*T, padding_mask
 * [B,T] or NULL.  Packed ragged batches (impl 1 only): cu_rows int32 [B+1] first row of every clip, T = longest clip.
 * impl 0 = mma.sync kernel, 1 = tcgen05 / TMEM kernel.  Replaces the attention inside
 * F.multi_head_attention_forward (fairseq/fairseq/modules/multihead_attention.py:170-192). */
AVH_API int avh_attention_bf16(const void* qkv, const uint8_t* padding_mask, const int32_t* cu_rows, int64_t rows, int B,
                               int T, int D, int H, int impl, void* out, void* stream);

/* Bare tcgen05 GEMM for kernel-level tests and profiling: C[M,N] = A[M,K] * B[N,K]^T (+bias)(gelu)(+R).
 * A,B bf16 row-major (K contiguous, K % 8 == 0), bias fp32 [N] or NULL, R/C bf16 or fp32 [M,N].
 * block_n: 0 = auto, else a multiple of 32 <= 256; pair: 0 = default, 1 = single-CTA tiles, 2 = CTA-pair tiles;
 * occ: 0 = auto, 1 = one CTA per SM, 2 = two CTAs per SM (block_n <= 128). */
AVH_API int avh_gemm_bf16(const void* A, const void* B, int64_t M, int N, int K, const float* bias, int gelu,
                  const void* R, int r_fp32, void* C, int c_fp32, int block_n, int pair, int occ, void* stream);

/* Debug: when dev_buf (device, >= 16*grid u64) is non-NULL every GEMM launch stamps %globaltimer at its
 * pipeline milestones per CTA; NULL switches it off. */
AVH_API int avh_gemm_set_trace(void* dev_buf);

/* Per-kernel-class timing of one forward for bench.py / profiles: with profiling on, avh_forward brackets
 * every launch with CUDA events on the launching stream; avh_profile_json waits for them and writes
 * {"class": {"launches": n, "ms": t, "tc_flops": executed tensor-core FLOPs}, ...} for the last forward. */
AVH_API int avh_set_profiling(avh_handle* h, int on);
AVH_API int avh_profile_json(avh_handle* h, char* buf, int64_t cap);

/* Counters for bench.py: kernels launched by this library since the last reset. */
AVH_API int64_t avh_launch_count(void);
AVH_API void avh_reset_launch_count(void);
/* CUDA-graph launches issued by the library since the process started (a forward replays 2-3 graph segments). */
AVH_API int64_t avh_graph_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* AVH_B200_H_ */
