// Internal launchers for the non-GEMM kernels of the AV-HuBERT hot path (all enqueue on `stream`,
// return 0 on success / 1 with avh::set_last_error on failure).
#pragma once
#include <cuda_runtime.h>
#include <vector_types.h>
#include <stdint.h>

namespace avh {

enum { DT_F32 = 0, DT_F16 = 1, DT_BF16 = 2 };

// Self-attention core on the fused QKV projection [B*T, 3*D] -> context [B*T, D]; bf16 or fp32 I/O.
// lse (optional, training): fp32 [B, H, T] log-sum-exp of every query row's scores
int launch_attention(const void* qkv, const unsigned char* kpm, void* out, int B, int T, int D, int H, int fp32,
                     cudaStream_t stream, float* lse = nullptr);
// backward of the above in bf16 mode (mma.sync): dO, O bf16 [B*T, D]; dqkv bf16 [B*T, 3*D] (dQ | dK | dV); Dbuf scratch [B,H,T]
int launch_attention_bwd_tc(const void* qkv, const void* dO, const void* O, const float* lse, const unsigned char* kpm,
                            void* dqkv, float* Dbuf, int B, int T, int D, int H, cudaStream_t stream);

// LayerNorm over the last dim C of [rows, C] (row stride ld_in); optional fp32 and low-precision outputs
// (both dense [rows, C]); rows flagged in row_zero (may be null) are written as zeros.
int launch_layernorm(const void* in, int in_dt, long long ld_in, const float* gamma, const float* beta, float eps,
                     float* out_f32, void* out_lp, int lp_dt, const unsigned char* row_zero, long long rows, int C,
                     cudaStream_t stream);

// generic strided [B, C, T] (any float dtype) -> row-major [B*T, ldo] (fp32/fp16/bf16): the
// x.transpose(1,2) in SubModel.forward (avhubert/hubert.py:327)
int launch_bct_to_rows(const void* in, int in_dt, long long sb, long long sc, long long st, int B, int C, int T,
                       void* out, int out_dt, long long ldo, cudaStream_t stream);

// ---- packed ragged batches: clips back to back, cu[b] = first row of clip b (device int32 [B+1])
int launch_bct_to_rows_ragged(const void* in, int in_dt, long long sb, long long sc, long long st, int B, int C,
                              const int* cu, void* out, int out_dt, long long ldo, long long rows_cap, cudaStream_t stream);
int launch_pos_pad_ragged(const float* in, long long ld, void* out, int* row_map, const int* cu, int B, int cols, int gap,
                          long long rows_pad, cudaStream_t stream);
int launch_unpack_rows(const float* in, const int* cu, void* out, int out_dt, int B, int T, int cols, cudaStream_t stream);

// [rows, cols] (fp32 / fp16 / bf16) -> fp32, rows flagged in row_zero (may be null) zeroed: index_put(x, padding_mask, 0)
int launch_load_rows(const void* in, int in_dt, float* out, const unsigned char* row_zero, long long rows, int cols,
                     cudaStream_t stream);
// per-sample linear resize along time of x [B,T,C] to len_out[b] rows (ATen upsample_linear1d arithmetic), zero tail, mask
int launch_interp_linear(const void* x, int dt, int B, int T, int C, const int* len_in, const int* len_out, int Tout,
                         void* out, long long* mask, cudaStream_t stream);
// flat element-wise dtype conversion
int launch_convert(const void* in, int in_dt, void* out, int out_dt, long long n, cudaStream_t stream);

// fp32 [rows, cols] (row stride ld) -> bf16 [rows', planes*cols]: plane 0 = round-to-nearest bf16 ("hi"),
// plane 1 = bf16 of the residual ("mid").  Optional time padding: out row = (r / T) * Tpad + r % T (T = 0:
// identity) — the zero-gapped token layout the positional convolution reads.
int launch_split_rows(const float* in, long long ld, void* out, int planes, long long rows, int cols, int T,
                      int Tpad, cudaStream_t stream);

// ---- lip frontend helpers (avhubert/resnet.py) ----------------------------------------------------
// spatial (kh,kw) patches of the 5x7x7/stride(1,2,2)/pad(2,3,3) stem for clips [b0, b0+nb): out bf16
// [nb*(T+2)*1936, planes*64], row = (bl*(T+2)+t)*1936 + pixel, column = kh*7+kw (49..63 zero; the two gap
// frames after each clip are left untouched = zero); planes = 2 adds the bf16 residual plane.
int launch_stem_patches(const void* video, int in_dt, int T, int b0, int nb, void* out, int planes,
                        cudaStream_t stream);
// MaxPool (1,3,3)/(1,2,2)/(0,1,1): NHWC frames [.,44,44,64] stored with two gap frames after every T frames
// (frame f at index (f/T)*(T+2) + f%T) -> zero-padded layout [nf,23,23,64] (bf16 or fp32)
int launch_maxpool_stem(const void* in, void* out, int nf, int T, int fp32, cudaStream_t stream);
// im2col for 3x3 stride-2 pad-1 convs reading the zero-padded bf16 layout [n,H+1,W+1,C] -> dense
// [n*Ho*Wo, 9*C] (K index = (kh*3+kw)*C + c)
int launch_im2col_s2(const void* in, void* out, int n, int H, int W, int C, cudaStream_t stream);
// mean over the H*W valid pixels of the padded layout [n,H+1,W+1,C] -> [n, C] (bf16 or fp32 in and out)
// raw uint8 gray frames [n, src_h, src_w] -> /255, centre crop, (x - mean) / std (avhubert/utils.py:56-95); frames
// flagged in frame_zero ([n], may be null: the key-padding mask) are written as 0.0, as the collater's zero padding is
int launch_video_preprocess(const unsigned char* frames, long long n_frames, int src_h, int src_w, int crop, double mean,
                            double stdv, void* out, int out_dt, const unsigned char* frame_zero, cudaStream_t stream);
int launch_avgpool(const void* in, void* out, int n, int H, int W, int C, int pitch, int fp32, cudaStream_t stream);

// ---- training-mode forward (train_ops.cu): BatchNorm with batch statistics, Philox dropout
constexpr int BN_SLOTS = 16;     // `sums` of bn_stats / bn_finalize holds BN_SLOTS x 2 x C doubles (zero before the first use)
int launch_bn_stats(const void* raw, int dt, long long rows, int C, long long period, long long valid, int S, int H,
                    double* sums, cudaStream_t stream);
int launch_bn_finalize(double* sums, double count, const float* gamma, const float* beta, float eps, float momentum,
                       float* rmean, float* rvar, float* scale, float* bias, int C, cudaStream_t stream);
int launch_bn_apply(const void* raw, void* out, int dt, long long rows, int C, const float* scale, const float* bias,
                    const float* slope1, const void* res, const float* slope2, int S, int H, cudaStream_t stream);
// x = dropout(x) in place (any dtype), or x += dropout(add) (fp32); mask = Philox4x32-10(seed, site, element)
int launch_dropout(void* x, int dt, const float* add, long long n, float p, unsigned long long seed, unsigned int site,
                   cudaStream_t stream);
// ---- dropout of the training step (train_dropout.cu): the same masks, the seed read from DEVICE memory (`seed`),
// 0 < p < 1, n and C multiples of 4; dtypes fp32 / bf16
// out = m * ((res ? res : 0) + gelu(u))
int launch_masked_gelu(const void* u, int u_dt, const float* res, void* out, int out_dt, long long n, float p,
                       const unsigned long long* seed, unsigned int site, cudaStream_t stream);
// y = (r ? r : 0) + m * a (fp32; y may alias a)
int launch_dropout_residual(const float* r, const float* a, float* y, long long n, float p, const unsigned long long* seed,
                            unsigned int site, cudaStream_t stream);
// du = m * dg * gelu'(u)
int launch_masked_gelu_bwd(const void* u, int u_dt, const void* dg, int dg_dt, void* du, int du_dt, long long n, float p,
                           const unsigned long long* seed, unsigned int site, cudaStream_t stream);
// out = m * dx over [rows, C] fp32 (out may alias dx); op != null: also its GEMM operand form (bf16 [rows, planes * C])
int launch_dropout_grad(const float* dx, float* out, void* op, int planes, long long rows, int C, float p,
                        const unsigned long long* seed, unsigned int site, cudaStream_t stream);

// ---- pretraining-mode extras (pretrain_ops.cu): span-mask substitution, masked-prediction logits, features_pen
// out unit u ([units, U] contiguous) = in unit code[u] (>= 0) | own (-1) | zeros (-2) | emb (-3); chan_zero [units / T, U]
int launch_mask_units(const void* in, void* out, int dt, const int* code, const void* emb, int emb_dt, long long units,
                      int U, const unsigned char* chan_zero, int T, cudaStream_t stream);
// the same on a strided [B,C,T] tensor (code per (b, t)), contiguous [B,C,T] out
int launch_mask_bct(const void* in, int dt, long long sb, long long sc, long long st, void* out, int out_dt,
                    const int* code, const void* emb, int emb_dt, int B, int C, int T, cudaStream_t stream);
// out[m,v] = (<F_m, E_v> + bias[v]) * inv_temp (mode 0) or / max(|F_m| |E_v|, 1e-6) * inv_temp (mode 1), fp32
int launch_logits(const void* F, int f_dt, long long ldf, const void* E, int e_dt, long long lde, const float* bias,
                  float* out, long long ldo, long long M, int V, int K, int mode, float inv_temp, cudaStream_t stream);
// its backward from the forward's logits and dL/dlogits [M,V] (row stride ldo): dF [M,K] (ldd_f), dE [V,K] (ldd_e), dbias [V]
// (each may be null), fp32; scratch: logits_bwd_scratch_floats(M, V, K) floats
int launch_logits_bwd(const void* F, int f_dt, long long ldf, const void* E, int e_dt, long long lde, long long M, int V, int K,
                      int mode, float inv_temp, const float* logits, const float* dlogits, long long ldo, float* dF, long long ldd_f,
                      float* dE, long long ldd_e, float* dbias, float* scratch, cudaStream_t stream);
long long logits_bwd_scratch_floats(long long M, int V, int K);
// dx[i] += dpen[0] * scale * x[i] (dpen: a device word)
int launch_pen_grad(const float* x, float* dx, long long n, const float* dpen, float scale, cudaStream_t stream);
// *acc = sum of squares of x (float64; acc is zeroed first)
int launch_sumsq(const void* x, int dt, long long n, double* acc, cudaStream_t stream);

// ---- Q-Former (qformer.cu): softmax(scale Q K^T + key mask) V with separate Q / K / V matrices (row strides in elements),
// head dim 64, heads side by side in the columns; key_pad [B, Lk] (1 = masked) or null; any float dtype in, o_dt out
int launch_attention_x(const void* Q, long long ldq, const void* K, long long ldk, const void* V, long long ldv, int dt,
                       const unsigned char* key_pad, void* O, long long ldo, int o_dt, int B, int H, int Lq, int Lk,
                       float scale, cudaStream_t stream, float* lse = nullptr);      // lse [B, H, Lq]: log-sum-exp per query row
// dst [B, per_clip] = src [per_clip] for every clip (fp32)
int launch_rows_broadcast(const float* src, float* dst, long long per_clip, int B, cudaStream_t stream);

// ---- backward of the Transformer encoder (backward_ops.cu)
// in [rows, C] -> bf16 [C, planes * kpad] (transposed GEMM operand over K = rows, zero padded), values times `scale`
// T > 0: K index (b * Tp + t) holds input row b * T + t, the gaps t in [T, Tp) are zeros (the positional conv's layout)
int launch_transpose_split(const void* in, int dt, long long ld, long long rows, int C, void* out, int planes, long long kpad,
                           float scale, cudaStream_t stream, int T = 0, int Tp = 0, long long out_ld = 0);      // out_ld: row stride
                                                                                    // of `out` when it differs from planes * kpad
int launch_scale(float* p, long long n, float s, cudaStream_t stream);
// positional-conv weight gradient helpers: shifted copies of the transposed input for one group; weight-norm backward
int launch_posconv_shift(const void* XT, void* XS, int g, int cg, int KT, int planes, long long kp, cudaStream_t stream);
int launch_posconv_weightnorm_bwd(const float* dw, const float* v, const float* g, int D, int cg, int KT, float* dg, float* dv,
                                  float* norms, cudaStream_t stream);
// out[c] = scale * sum_r in[r, c]  (bias gradients)
int launch_colsum(const void* in, int dt, long long ld, long long rows, int C, float* out, float scale, cudaStream_t stream);
// out = (res ? res : 0) + gelu(u);  du = dg * gelu'(u)
int launch_gelu_fwd(const void* u, int u_dt, const float* res, void* out, int out_dt, long long n, cudaStream_t stream);
int launch_gelu_bwd(const void* u, int u_dt, const void* dg, int dg_dt, void* du, int du_dt, long long n, cudaStream_t stream);
// LayerNorm backward: dx_out = (res ? res : 0) + dLN/dx(dy), dgamma, dbeta; stats = scratch [rows] float2
int launch_ln_bwd(const float* x, const float* gamma, const float* dy, const float* res, float* dx_out, float2* stats,
                  float* dgamma, float* dbeta, long long rows, int C, float eps, cudaStream_t stream);
// post-LN LayerNorm backward: dx_out = dLN/dx(dya + dyb) (dyb may be null), dgamma / dbeta of the summed gradient;
// v = m * dx_out with m the dropout mask of `site` (p = 0: v = dx_out; p > 0: seed is a DEVICE word) into mout (fp32,
// optional) and op (GEMM operand form, bf16 [rows, planes * C]); C a multiple of 4; outputs must not alias dya / dyb
int launch_ln_post_bwd(const float* x, const float* gamma, const float* dya, const float* dyb, float* dx_out, float* mout,
                       void* op, int planes, float2* stats, float* dgamma, float* dbeta, long long rows, int C, float eps,
                       float p, const unsigned long long* seed, unsigned int site, cudaStream_t stream);
// attention backward (self-attention over L rows per clip, heads of 64 channels side by side); Dbuf = scratch [B, H, L]
int launch_attention_bwd(const void* Q, long long ldq, const void* K, long long ldk, const void* V, long long ldv, int dt,
                         const void* dO, const void* O, long long ldo, int o_dt, const float* lse, const unsigned char* key_pad,
                         void* dQ, void* dK, void* dV, long long ldd, int d_dt, float* Dbuf, int B, int H, int L,
                         cudaStream_t stream);

// ---- training step of the lip ResNet on dense NHWC maps (frontend_train.cu)
int launch_im2col_stem(const void* video, int dt, int B, int T, void* col, int planes, cudaStream_t stream);
int launch_im2col2d(const void* x, int dt, long long n, int H, int C, int ks, int stride, int pad, int Ho, void* col, int planes,
                    cudaStream_t stream);
// ---- refresh.cu: packed weights rewritten in place from device-resident parameters (index maps of api.cu's packers)
int launch_refresh_matrix(const void* src, int dt, long long n, long long k, float scale, void* dst, long long ld, int planes,
                          long long off, int transposed, cudaStream_t stream);
int launch_refresh_vec(const void* src, int dt, long long n, long long n_src, float scale, float* dst, cudaStream_t stream);
int launch_refresh_conv(const void* src, int dt, int cout, int cin, int ksq, void* dst, long long ld, int planes, int transposed,
                        cudaStream_t stream);
int launch_refresh_stem(const void* src, int dt, void* dst, int planes, int pitch8, cudaStream_t stream);
int launch_posconv_ratio(const void* v, int v_dt, const void* g, int g_dt, long long per_tap, int KT, float* ratio,
                         cudaStream_t stream);
int launch_refresh_pos(const void* v, int dt, const float* ratio, const int* acol, int D, int cg, int KT, int window, void* dst,
                       int planes, int transposed, cudaStream_t stream);
// eval-only forms: the BatchNorm fold (scale / bias, and the fp32 gamma / beta / running statistics) and the conv2 +
// shortcut GEMM weights with both BatchNorm scales folded in, bit-identical to the host packers
int launch_bn_fold(const void* g, int g_dt, const void* b, int b_dt, const void* m, int m_dt, const void* v, int v_dt, int C,
                   float* scale, float* bias, float* gamma, float* beta, float* rmean, float* rvar, cudaStream_t stream);
int launch_refresh_c2ds(const void* w2, int w2_dt, const void* wd, int wd_dt, const float* s2, const float* b2, const float* sd,
                        const float* bd, int cout, int cmid, int cin, void* dst, int planes, float* bias, cudaStream_t stream);
int launch_im2colT(const void* x, long long n, int H, int C, int ks, int stride, int pad, int Ho, void* colT, long long kp,
                   cudaStream_t stream);          // bf16 x -> bf16 colT [ks*ks*C, kp] (transposed patches)
int launch_transposeT(const void* in, int dt, long long ld, long long rows, int C, void* out, long long kp, long long out_ld,
                      cudaStream_t stream, float scale = 1.0f);       // [rows, C] bf16 / fp32 -> bf16 [C, out_ld] (64 x 64 tiles)
int launch_col2im2d(const void* dcol, int dt, long long n, int H, int C, int ks, int stride, int pad, int Ho, float* dx,
                    int accumulate, cudaStream_t stream);
int launch_maxpool_dense(const void* x, void* y, int dt, long long n, int H, int C, int Ho, cudaStream_t stream,
                         unsigned char* arg = nullptr);     // arg: window position of every maximum (bf16 maps), for the backward
int launch_maxpool_bwd(const void* x, int dt, const float* dy, float* dx, long long n, int H, int C, int Ho, cudaStream_t stream,
                       const unsigned char* arg = nullptr);
int launch_avgpool_dense(const void* x, void* y, int dt, long long n, int HW, int C, cudaStream_t stream);
int launch_avgpool_bwd(const float* dy, float* dx, long long n, int HW, int C, cudaStream_t stream);
// stat [2*C] = batch mean, rstd recovered from bn_finalize's (scale, bias)
int launch_bn_stat_from_affine(const float* scale, const float* bias, const float* gamma, const float* beta, int C, float* stat,
                               cudaStream_t stream);
// BatchNorm(batch stats) [+ residual] [+ PReLU] backward on [rows, C]: d_raw, d_res (optional, = or +=), dgamma, dbeta, dslope;
// sums = BN_SLOTS x 3 x C doubles (zero before the first use), tot = 3 x C floats scratch
int launch_bn_act_bwd(const void* raw, int dt, const void* res, const float* dz, const float* stat, const float* gamma,
                      const float* beta, const float* slope, long long rows, int C, double* sums, float* tot, void* d_raw,
                      float* d_res, int res_accumulate, float* dgamma, float* dbeta, float* dslope, cudaStream_t stream,
                      int d_raw_dt = DT_F32);       // d_raw_dt = DT_BF16 (bf16 maps only): the map gradient as a GEMM operand
int launch_add_f32(float* a, const float* b, long long n, cudaStream_t stream);

// ---- audio frontend ---------------------------------------------------------------------------------
struct FbankArgs {
  const int16_t* wav;          // concatenated clips
  const long long* offsets;    // [n_clips+1] sample offsets (device)
  const int* video_len;        // [n_clips] frames to align to, or null (use own stacked length)
  int n_clips;
  int T;                       // output rows per clip (collated size)
  int normalize;               // per-row LayerNorm over the 104 features
  float* out;                  // [n_clips, T, 104]
  unsigned char* padding_mask; // [n_clips, T] or null
};
int launch_fbank(const FbankArgs& a, cudaStream_t stream);
// hubert_dataset.py:317-346 on device: mixed int16 = trunc(clip_rescale(clean + noise * scale))
int launch_add_noise(const int16_t* clean, const long long* offsets, int n_clips, const float* noise,
                     long long noise_len, float snr_db, int16_t* out, double* scratch, cudaStream_t stream);

}  // namespace avh
