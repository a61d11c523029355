// Internal C++ interface of the tcgen05 GEMM ("shifted-row multi-tap GEMM") used by every dense
// contraction on the AV-HuBERT path: Linear layers, the grouped positional conv, 3x3/1x1 convs of the
// lip ResNet (implicit GEMM over a zero-padded NHWC layout) and the bf16x3 split-precision fp32 mode.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <vector_types.h>
#include <stdint.h>

#include <vector>

namespace avh {

enum { ACT_NONE = 0, ACT_GELU = 1, ACT_PRELU = 2 };
enum { MAP_IDENTITY = 0, MAP_2LEVEL = 1 };

// out = rowmask( act2( act1( acc * col_scale + col_bias ) + R ) ), written as bf16 or fp32.
struct Epilogue {
  void* C = nullptr;
  long long ldc = 0;
  int c_fp32 = 0;
  const float* col_scale = nullptr;
  const float* col_bias = nullptr;
  int act = ACT_NONE;
  const float* slope1 = nullptr;        // PReLU slopes (per column) for act
  const void* R = nullptr;              // residual, same row mapping as C
  long long ldr = 0;
  int r_fp32 = 0;
  const float* slope2 = nullptr;        // PReLU applied after the residual add
  const unsigned char* row_zero = nullptr;  // [out rows] 1 -> row forced to 0 (key-padding mask)
  // tile row r -> output row.  MAP_2LEVEL: n=r/S2, rem=r%S2, h=rem/S1, w=rem%S1,
  // valid = h<H && w<W, out_row = n*O2 + h*O1 + w + O0.
  int map_mode = MAP_IDENTITY;
  int S1 = 1, S2 = 1, H = 1, W = 1;
  long long O0 = 0, O1 = 0, O2 = 0;
  int invalid_zero = 0;                 // invalid rows: 1 -> store zeros, 0 -> skip
  const int* row_map = nullptr;         // device [M]: tile row -> output row, -1 = skip (overrides map_mode; ragged pos-conv)
};

// One K-block (64 bf16 along K) of the contraction: A box at (col, m0 + row_off), B box at (col, n0 + row_off).
struct KStep {
  int a_col, a_row_off, b_col, b_row_off;
};

struct GemmProblem {
  const void* A = nullptr;  // bf16 [a_rows, a_cols], row stride lda (elements, multiple of 8)
  long long a_rows = 0;
  int a_cols = 0;
  long long lda = 0;
  const void* B = nullptr;  // bf16 [b_rows, b_cols], row stride ldb
  long long b_rows = 0;
  int b_cols = 0;
  long long ldb = 0;
  long long M = 0;          // tile-row space size
  int N = 0;                // output columns (multiple of 32)
  int num_kb = 0;           // number of K blocks
  const KStep* ktable = nullptr;  // device pointer, num_kb entries; null -> a_col=b_col=kb*64, offsets 0
  int a_col_per_nblk = 0;   // grouped conv: A column offset added per N tile
  const int* a_col_nblk = nullptr;  // device table [num N tiles] of A column offsets (overrides a_col_per_nblk)
  int block_n = 0;          // output-tile width: multiple of 32, <= 256; 0 = chosen by gemm_plan (wave fitting)
  int occ = 0;              // CTAs per SM: 0 = chosen by gemm_plan, 1, or 2 (block_n <= 128 only)
  int pair = 0;             // 0 = default (CTA pairs, tcgen05 cta_group::2), 1 = single-CTA form, 2 = pairs
  // stream-K workspace (optional): fp32 partial accumulators [units][pair * 128][block_n] + one flag per CTA, zeroed
  // once by the owner of the buffers.  With it, gemm_plan may cut the tile x k-block space into equal ranges per unit
  // instead of whole tiles (deterministic: fixed partition, partials added in unit order).
  float* sk_ws = nullptr;
  size_t sk_ws_bytes = 0;
  int* sk_flags = nullptr;  // >= 2 * SMs ints
  int streamk = 0;          // 0 = gemm_plan decides (needs the workspace), 1 = force on, -1 = off
  Epilogue ep;
};

struct GemmPlan {
  CUtensorMap tma_a, tma_b, tma_c;
  int c_mode = 0;
  int sk = 0;                     // stream-K partition in use
  GemmProblem prob;
  int grid = 0;
  int stages = 0;
  int ktab_bytes = 0;
  size_t smem = 0;
};

// ---- 3x3 / stride-1 / 64 -> 64 channel convolution over the shared-zero-padded NHWC layout with the operand
// window resident in smem: ONE TMA load of 128 + 2(S+1) rows per tile, the nine taps are tcgen05.mma operand
// descriptors that start at different ROWS of that window (the 128-byte swizzle is a function of the absolute
// smem address, so a descriptor may start at any row: tools/micro/desc_offset.cu), all 9 x 64 x 64 weights stay
// resident in smem.  Cuts the L2->SM operand stream of the layer1 convolutions ~9x.
struct ConvWinProblem {
  const void* A = nullptr;        // bf16 [rows, 64] padded layout, flat
  const void* B = nullptr;        // bf16 [64, 9*64] K-major weights, K = (tap, cin)
  long long rows = 0;             // n * S * S
  int S = 0;                      // padded image pitch (H + 1); H = W = S - 1 valid rows/columns
  const float* scale = nullptr;   // folded BatchNorm
  const float* bias = nullptr;
  const float* slope1 = nullptr;  // PReLU before the residual (conv1) or null
  const void* R = nullptr;        // bf16 residual [rows, 64] or null
  const float* slope2 = nullptr;  // PReLU after the residual (conv2) or null
  void* C = nullptr;              // bf16 [rows, 64]
};
struct ConvWinPlan {
  CUtensorMap tma_a, tma_b, tma_c;
  ConvWinProblem prob;
  int grid = 0, stages = 0, win_rows = 0;
  size_t smem = 0;
};
int conv_window_plan(const ConvWinProblem& prob, ConvWinPlan* plan);
int conv_window_launch(const ConvWinPlan& plan, cudaStream_t stream);
// ---- convolutions of the small maps (layers 2-4) with one frame per GEMM row: activations [frames, P*C],
// tile = 128 frames x block_n channels of one output pixel, K loop = in-image taps only (conv_frame.cu).
struct ConvFrameProblem {
  const void* A = nullptr;        // bf16 [frames, Pin*Cin]
  long long frames = 0;
  int Hin = 0, Sin = 0, Pin = 0, Cin = 0;      // input image H = W, pixel pitch, pixels per frame row, channels
  const void* B = nullptr;        // bf16 [Cout, ks*ks*Cin] K-major weights, K = (tap, cin)
  int Cout = 0, ks = 3, stride = 1;            // padding = 1 for ks 3, 0 for ks 1
  int Hout = 0, Sout = 0, Pout = 0;            // output image, pitch, pixels per frame row
  const float* scale = nullptr;   // folded BatchNorm
  const float* bias = nullptr;
  const float* slope1 = nullptr;  // PReLU (conv1 form) or null
  const void* R = nullptr;        // bf16 residual in the output layout (conv2 form) or null
  const float* slope2 = nullptr;  // PReLU after the residual add
  void* C = nullptr;              // bf16 [frames, Pout*Cout]
  // optional fused 1x1 stride-s shortcut conv (downsample_basic_block, resnet.py:20-24) accumulated into the same
  // tile: second input A2 [frames, ds_Pin*ds_Cin] (pixel pitch ds_Sin), sampled at (oy*ds_stride, ox*ds_stride);
  // its weights are the columns [ks*ks*Cin, +ds_Cin) of B.  Both BatchNorm scales must be folded into B then.
  const void* A2 = nullptr;
  int ds_Cin = 0, ds_Sin = 0, ds_Pin = 0, ds_stride = 1;
  int block_n = 0, occ = 0;       // 0 = chosen by conv_frame_plan
  int pair = 0;                   // 0 = default (CTA pairs where the tile allows), 1 = single CTAs, 2 = pairs
};
struct ConvFramePlan {
  CUtensorMap tma_a, tma_b, tma_c, tma_a2;
  ConvFrameProblem prob;
  int grid = 0, stages = 0, pair = 1;
  size_t smem = 0;
  std::vector<int> tiles_host;    // [grid+1] offsets + per-CTA tile lists
  const int* tiles_dev = nullptr;
};
int conv_frame_plan(const ConvFrameProblem& prob, ConvFramePlan* plan);
size_t conv_frame_table_bytes(const ConvFrameProblem& prob);        // device bytes to reserve for the tile table
int conv_frame_bind_table(ConvFramePlan* plan, void* dev_table);    // uploads the table (synchronous copy)
int conv_frame_launch(const ConvFramePlan& plan, cudaStream_t stream);
// ---- fused lip-frontend stem: Conv3d 5x7x7 + BN + PReLU + MaxPool in one kernel (stem_fused.cu)
struct StemFusedPlan {
  const void* w = nullptr;        // weights bf16 [64, 5*64], K = dt*64 + kh*8 + kw (kw = 7 and k >= 56 zero)
};
int stem_fused_plan(const void* w_packed, StemFusedPlan* plan);
int stem_fused_launch(const StemFusedPlan& plan, const void* video, int in_dt, int T, int b0, int nb, const float* scale,
                      const float* bias, const float* slope, void* pooled_out, cudaStream_t stream);
// ---- self-attention on tcgen05 / TMEM (attention_tc.cu): S = Q K^T and O = P V as UMMAs, P read from tensor memory
struct AttnTcPlan {
  CUtensorMap tma_q, tma_kv;      // boxes of 128 / kv_rows rows x 64 columns over the QKV matrix [rows, 3*D]
  int B = 0, T = 0, D = 0, H = 0;
  int kv_rows = 0, stages = 0, stage_bytes = 0, mask_floats = 0;
  size_t smem = 0;
};
int attention_tc_plan(const void* qkv, long long rows, int B, int T, int D, int H, AttnTcPlan* plan);
// kpm: [B, T] key-padding mask or null; cu: [B + 1] first row of every clip for packed ragged batches, or null
int attention_tc_launch(const AttnTcPlan& plan, const unsigned char* kpm, const int* cu, void* out, cudaStream_t stream);
// ragged batches (clips of different lengths packed back to back in the output): host-built work list + launch
int stem_fused_ragged_items(const int* lengths, int n_clips, int sms, int4* items, int max_items);   // returns count or -1
int stem_fused_launch_ragged(const StemFusedPlan& plan, const void* video, int in_dt, int Tpitch, const int4* items,
                             const int* n_items, const int* cu, const float* scale, const float* bias, const float* slope,
                             void* out, cudaStream_t stream);
// tensor-map helpers shared by the GEMM kernels (gemm_tcgen05.cu)
int encode_2d(CUtensorMap* map, const void* base, long long rows, int cols, long long ld, int box_rows);
int encode_c(CUtensorMap* map, const void* base, long long rows, int cols, long long ld, int fp32);

constexpr int GEMM_MAX_KSTEPS = 768;

int gemm_plan(const GemmProblem& prob, GemmPlan* plan);       // builds tensor maps; 0 on success
int gemm_launch(const GemmPlan& plan, cudaStream_t stream);  // enqueue; 0 on success
void gemm_set_trace(unsigned long long* dev_buf);             // debug: per-CTA globaltimer stamps [grid][16]

}  // namespace avh
