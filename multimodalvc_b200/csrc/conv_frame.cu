// Convolutions of the small feature maps of the lip ResNet (layers 2-4: 11x11x128, 6x6x256, 3x3x512; 3x3 stride 1,
// 3x3 stride 2 and the 1x1 stride-2 downsample, + folded BatchNorm, PReLU, residual, PReLU) on tcgen05 with ONE
// FRAME PER GEMM ROW (avhubert/resnet.py:35-74,99-129).
//
// Layout: an activation is [frames, P * C] bf16 — row = frame, column = (pixel, channel), pixel = y * pitch + x.
// The layer1 output keeps its shared-zero-padded 23 x 23 pitch (it is written by conv_window.cu); layers 2-4 are
// dense (pitch = H).  An output tile is 128 frames x BN channels of ONE output pixel (oy, ox); its K loop walks
// only the taps that fall inside the image: A box = 128 frames x 64 channels of input pixel
// (oy*stride + kh - pad, ox*stride + kw - pad) — a column offset into the frame rows —, B box = the 64-channel slice
// of tap (kh, kw).  Compared with the shifted-row implicit GEMM over a zero-padded map this spends no MMAs on pad
// pixels or out-of-image taps ((H+1)^2 * 9 -> (3H-2)^2 tap-pixels: 1.35x fewer for 11x11, 1.7x for 6x6, 2.9x for
// 3x3), needs no im2col for stride 2, and writes dense maps.
//
// Tiles differ in cost (4, 6 or 9 taps), so the host assigns them to CTAs with a longest-processing-time greedy
// pass over groups of frame blocks (a group's input stays in L2 while its pixels are processed) and hands the kernel
// per-CTA tile lists.  Roles as in gemm_tcgen05.cu: warp 0 TMA producer, warp 1 MMA issuer (elected lane,
// warp-uniform loops), warp 2 TMEM allocator, warps 4.. epilogue (thread = frame row: tcgen05.ld ->
// scale/bias/PReLU/residual/PReLU -> swizzled smem box -> TMA store).  OCC = 2 (two CTAs per SM, BN = 128) for the
// 128-channel layer, OCC = 1 with BN = 256 for the wider ones.
#include "common.cuh"
#include "gemm.h"

#include <algorithm>
#include <cstdlib>
#include <mutex>
#include <set>
#include <vector>

namespace avh {
namespace {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int A_STAGE_BYTES = BM * BK * 2;
constexpr int MAX_STAGES = 8;
constexpr int MAX_COUT = 512;
constexpr int COLVEC_BYTES = 4 * MAX_COUT * 4;     // scale | bias | slope1 | slope2 for all output channels
constexpr int BAR_BYTES = (2 * MAX_STAGES + 4) * 8 + 16;

template <int OCC>
struct FOcc {
  static constexpr int EPI_WARPS = OCC == 2 ? 4 : 8;
  static constexpr int NUM_THREADS = 128 + 32 * EPI_WARPS;
  static constexpr int TMEM_COLS = 512 / OCC;
  static constexpr int ACC_STRIDE = 256 / OCC;
  static constexpr int EPI_STAGE_BYTES = EPI_WARPS * 4096;
  static constexpr int SMEM_LIMIT = OCC == 2 ? 113 * 1024 : 227 * 1024;
  static constexpr int HSTRIDE = EPI_WARPS / 4;
};

struct FrameParams {
  long long frames;
  int Hin, Sin, Cin;            // input image size, pixel pitch, channels
  int Hout, Sout, Cout;
  int ks, stride, pad;
  int block_n, stages;
  int chunks;                   // Cin / 64
  // fused 1x1 stride-s shortcut (downsample_basic_block): extra K steps over a SECOND input tensor, the pixel
  // (oy*ds_stride, ox*ds_stride) of it, against weight columns [ds_bcol, ds_bcol + ds_chunks*64)
  int ds_chunks, ds_stride, ds_Sin, ds_Cin, ds_bcol;
  long long ldr;                // residual row stride (elements) = output row stride
  const int* tiles;             // [grid + 1] offsets followed by the tile lists
  const float* scale;
  const float* bias;
  const float* slope1;
  const float* slope2;
  const __nv_bfloat16* R;
};

// tile code: frame block | oy << 16 | ox << 21 | n_sub << 26
__device__ __forceinline__ void decode_tile(int code, int& m_blk, int& oy, int& ox, int& nsub) {
  m_blk = code & 0xFFFF;
  oy = (code >> 16) & 31;
  ox = (code >> 21) & 31;
  nsub = (code >> 26) & 7;
}

// MODE 0: BN only (downsample), 1: BN + PReLU (conv1), 2: BN + residual + PReLU (conv2)
// PAIR 2: a cluster of two CTAs (the two SMs of a TPC) owns a 256-frame x BN tile and drives ONE
// tcgen05.mma.cta_group::2 per K step: each CTA stages its own 128 frames of A and HALF of the weight tile, so an SM
// pulls 16 KB + 64 BN B per k-block through its ~64 B/clk L2 ingress instead of 16 KB + 128 BN — the single-CTA tiles
// of these layers are bound by that ingress (785 clk per k-block at BN 256 against 512 clk of tensor work).
template <int OCC, int MODE, int PAIR>
__global__ void __launch_bounds__(FOcc<OCC>::NUM_THREADS, OCC)
conv_frame_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                  const __grid_constant__ CUtensorMap tma_c, const __grid_constant__ CUtensorMap tma_a2,
                  const FrameParams p) {
  constexpr int EPI_WARPS = FOcc<OCC>::EPI_WARPS;
  constexpr int NUM_THREADS = FOcc<OCC>::NUM_THREADS;
  constexpr int TMEM_COLS = FOcc<OCC>::TMEM_COLS;
  constexpr int ACC_STRIDE = FOcc<OCC>::ACC_STRIDE;
  constexpr int HSTRIDE = FOcc<OCC>::HSTRIDE;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  const int BN = p.block_n;
  const int STAGES = p.stages;
  const int b_stage_bytes = (BN / PAIR) * BK * 2;
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + STAGES * A_STAGE_BYTES;
  uint8_t* epi_stage = smem_b + STAGES * b_stage_bytes;
  float* colvec = reinterpret_cast<float*>(epi_stage + FOcc<OCC>::EPI_STAGE_BYTES);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(colvec) + COLVEC_BYTES);
  uint64_t* empty_bar = full_bar + MAX_STAGES;
  uint64_t* tmem_full = empty_bar + MAX_STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int cta_rank = PAIR == 2 ? (int)cluster_ctarank() : 0;
  const bool leader = cta_rank == 0;
  const int unit = blockIdx.x / PAIR;
  pdl_launch_dependents();

  // launch-constant data: per-channel vectors, this unit's tile list bounds
  for (int c = threadIdx.x; c < p.Cout; c += NUM_THREADS) {
    colvec[c] = __ldg(p.scale + c);
    colvec[MAX_COUT + c] = __ldg(p.bias + c);
    colvec[2 * MAX_COUT + c] = p.slope1 != nullptr ? __ldg(p.slope1 + c) : 1.f;
    colvec[3 * MAX_COUT + c] = p.slope2 != nullptr ? __ldg(p.slope2 + c) : 1.f;
  }
  const int t_begin = __ldg(p.tiles + unit);
  const int t_end = __ldg(p.tiles + unit + 1);
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
    tma_prefetch_desc(&tma_c);
    if (p.ds_chunks > 0) tma_prefetch_desc(&tma_a2);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], PAIR * EPI_WARPS);
    }
    mbar_fence_init();
  }
  if (warp == 2) {
    if (PAIR == 2) tmem_alloc_pair(tmem_slot, TMEM_COLS);
    else tmem_alloc(tmem_slot, TMEM_COLS);
  }
  tc_fence_before();
  if (PAIR == 2) cluster_sync_all();
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    int stage = 0;
    uint32_t phase = 0;
    const uint32_t stage_tx = (uint32_t)PAIR * (uint32_t)(A_STAGE_BYTES + b_stage_bytes);
    for (int ti = t_begin; ti < t_end; ++ti) {
      int m_blk, oy, ox, nsub;
      decode_tile(__ldg(p.tiles + ti), m_blk, oy, ox, nsub);
      const int m0 = (m_blk * PAIR + cta_rank) * BM, n0 = nsub * BN + cta_rank * (BN / PAIR);
      for (int kh = 0; kh < p.ks; ++kh) {
        const int iy = oy * p.stride + kh - p.pad;
        if (iy < 0 || iy >= p.Hin) continue;
        for (int kw = 0; kw < p.ks; ++kw) {
          const int ix = ox * p.stride + kw - p.pad;
          if (ix < 0 || ix >= p.Hin) continue;
          const int a_col = (iy * p.Sin + ix) * p.Cin;
          const int b_col = (kh * p.ks + kw) * p.Cin;
          for (int kc = 0; kc < p.chunks; ++kc) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            if (elect_one()) {
              if (leader) mbar_expect_tx(&full_bar[stage], stage_tx);
              if (PAIR == 2) {
                tma_load_2d_pair(smem_a + stage * A_STAGE_BYTES, &tma_a, &full_bar[stage], a_col + kc * BK, m0);
                tma_load_2d_pair(smem_b + stage * b_stage_bytes, &tma_b, &full_bar[stage], b_col + kc * BK, n0);
              } else {
                tma_load_2d(smem_a + stage * A_STAGE_BYTES, &tma_a, &full_bar[stage], a_col + kc * BK, m0);
                tma_load_2d(smem_b + stage * b_stage_bytes, &tma_b, &full_bar[stage], b_col + kc * BK, n0);
              }
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
      for (int kc = 0; kc < p.ds_chunks; ++kc) {          // fused shortcut: centre pixel of the block's input
        mbar_wait(&empty_bar[stage], phase ^ 1);
        if (elect_one()) {
          if (leader) mbar_expect_tx(&full_bar[stage], stage_tx);
          const int a2_col = ((oy * p.ds_stride) * p.ds_Sin + ox * p.ds_stride) * p.ds_Cin + kc * BK;
          if (PAIR == 2) {
            tma_load_2d_pair(smem_a + stage * A_STAGE_BYTES, &tma_a2, &full_bar[stage], a2_col, m0);
            tma_load_2d_pair(smem_b + stage * b_stage_bytes, &tma_b, &full_bar[stage], p.ds_bcol + kc * BK, n0);
          } else {
            tma_load_2d(smem_a + stage * A_STAGE_BYTES, &tma_a2, &full_bar[stage], a2_col, m0);
            tma_load_2d(smem_b + stage * b_stage_bytes, &tma_b, &full_bar[stage], p.ds_bcol + kc * BK, n0);
          }
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1 && leader) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA of a pair)
    const uint32_t idesc = umma_idesc_bf16(BM * PAIR, BN);
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int ti = t_begin; ti < t_end; ++ti, ++it) {
      int m_blk, oy, ox, nsub;
      decode_tile(__ldg(p.tiles + ti), m_blk, oy, ox, nsub);
      int ny = 0, nx = 0;
      for (int k = 0; k < p.ks; ++k) {
        const int iy = oy * p.stride + k - p.pad, ix = ox * p.stride + k - p.pad;
        ny += (iy >= 0 && iy < p.Hin) ? 1 : 0;
        nx += (ix >= 0 && ix < p.Hin) ? 1 : 0;
      }
      const int num_kb = ny * nx * p.chunks + p.ds_chunks;
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + acc * ACC_STRIDE;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint64_t adesc = umma_desc_sw128(smem_u32(smem_a + stage * A_STAGE_BYTES));
        const uint64_t bdesc = umma_desc_sw128(smem_u32(smem_b + stage * b_stage_bytes));
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            if (PAIR == 2) umma_bf16_pair(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0);
            else umma_bf16(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0);
          }
          if (PAIR == 2) umma_commit_pair(&empty_bar[stage]);      // smem slot reusable in BOTH CTAs
          else umma_commit(&empty_bar[stage]);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
      if (elect_one()) {
        if (PAIR == 2) umma_commit_pair(&tmem_full[acc]);
        else umma_commit(&tmem_full[acc]);
      }
      __syncwarp();
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ epilogue: thread = frame row
    const int q = warp & 3;
    const int half = (warp - 4) >> 2;
    uint8_t* stg = epi_stage + (warp - 4) * 4096;
    const int nboxes = BN / 64;
    int it = 0;
    for (int ti = t_begin; ti < t_end; ++ti, ++it) {
      int m_blk, oy, ox, nsub;
      decode_tile(__ldg(p.tiles + ti), m_blk, oy, ox, nsub);
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int row0 = (m_blk * PAIR + cta_rank) * BM + q * 32;
      const long long r = (long long)row0 + lane;
      const bool live = r < p.frames;
      const int ch0 = nsub * BN;                                   // first output channel of the tile
      const int ccol0 = (oy * p.Sout + ox) * p.Cout + ch0;         // first output column of the tile
      uint4 rres[8];
      if (MODE == 2 && live && half < nboxes) {                    // residual of the first box in flight early
        const uint4* rp = reinterpret_cast<const uint4*>(p.R + r * p.ldr + ccol0 + half * 64);
#pragma unroll
        for (int j = 0; j < 8; ++j) rres[j] = __ldg(rp + j);
      }
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * ACC_STRIDE;
#pragma unroll 1
      for (int bx = half; bx < nboxes; bx += HSTRIDE) {
        const int cbase = bx * 64;
        uint32_t packed[32];
#pragma unroll
        for (int sub = 0; sub < 2; ++sub) {
          const int c0 = cbase + sub * 32;
          uint32_t rawv[32];
          tmem_ld_32x32(taddr + c0, rawv);
          tmem_ld_wait();
          const float* cv = colvec + ch0 + c0;
          float v[32];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 sc = *reinterpret_cast<const float4*>(cv + 4 * j);
            const float4 bi = *reinterpret_cast<const float4*>(cv + MAX_COUT + 4 * j);
            v[4 * j] = fmaf(__uint_as_float(rawv[4 * j]), sc.x, bi.x);
            v[4 * j + 1] = fmaf(__uint_as_float(rawv[4 * j + 1]), sc.y, bi.y);
            v[4 * j + 2] = fmaf(__uint_as_float(rawv[4 * j + 2]), sc.z, bi.z);
            v[4 * j + 3] = fmaf(__uint_as_float(rawv[4 * j + 3]), sc.w, bi.w);
          }
          if (MODE == 1) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 s1 = *reinterpret_cast<const float4*>(cv + 2 * MAX_COUT + 4 * j);
              v[4 * j] = v[4 * j] > 0.f ? v[4 * j] : v[4 * j] * s1.x;
              v[4 * j + 1] = v[4 * j + 1] > 0.f ? v[4 * j + 1] : v[4 * j + 1] * s1.y;
              v[4 * j + 2] = v[4 * j + 2] > 0.f ? v[4 * j + 2] : v[4 * j + 2] * s1.z;
              v[4 * j + 3] = v[4 * j + 3] > 0.f ? v[4 * j + 3] : v[4 * j + 3] * s1.w;
            }
          }
          if (MODE == 2) {
            if (live) {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&rres[sub * 4 + j]);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const float2 f = __bfloat1622float2(h2[k]);
                  v[8 * j + 2 * k] += f.x;
                  v[8 * j + 2 * k + 1] += f.y;
                }
              }
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 s2 = *reinterpret_cast<const float4*>(cv + 3 * MAX_COUT + 4 * j);
              v[4 * j] = v[4 * j] > 0.f ? v[4 * j] : v[4 * j] * s2.x;
              v[4 * j + 1] = v[4 * j + 1] > 0.f ? v[4 * j + 1] : v[4 * j + 1] * s2.y;
              v[4 * j + 2] = v[4 * j + 2] > 0.f ? v[4 * j + 2] : v[4 * j + 2] * s2.z;
              v[4 * j + 3] = v[4 * j + 3] > 0.f ? v[4 * j + 3] : v[4 * j + 3] * s2.w;
            }
          }
#pragma unroll
          for (int j = 0; j < 16; ++j) packed[sub * 16 + j] = pack_bf16(v[2 * j], v[2 * j + 1]);
        }
        if (bx + HSTRIDE >= nboxes) {
          // last TMEM read of this accumulator stage by this warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (PAIR == 2) mbar_arrive_leader(&tmem_empty[acc]);
            else mbar_arrive(&tmem_empty[acc]);
          }
        } else if (MODE == 2 && live) {
          const uint4* rp = reinterpret_cast<const uint4*>(p.R + r * p.ldr + ccol0 + (bx + HSTRIDE) * 64);
#pragma unroll
          for (int j = 0; j < 8; ++j) rres[j] = __ldg(rp + j);
        }
        if (lane == 0) tma_wait_group_read0();
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 8; ++j)
          *reinterpret_cast<uint4*>(stg + lane * 128 + ((j ^ (lane & 7)) << 4)) =
              make_uint4(packed[4 * j], packed[4 * j + 1], packed[4 * j + 2], packed[4 * j + 3]);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0 && row0 < p.frames) {
          tma_store_2d(&tma_c, stg, ccol0 + cbase, row0);          // rows beyond the last frame are clipped by TMA
          tma_commit_group();
        }
      }
      if (half >= nboxes) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (PAIR == 2) mbar_arrive_leader(&tmem_empty[acc]);
          else mbar_arrive(&tmem_empty[acc]);
        }
      }
    }
    if (lane == 0) tma_wait_group0();
  }

  tc_fence_before();
  if (PAIR == 2) cluster_sync_all();
  else __syncthreads();
  tc_fence_after();
  if (warp == 2) {
    if (PAIR == 2) tmem_dealloc_pair(tmem_base, TMEM_COLS);
    else tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

typedef void (*FrameKernelFn)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, FrameParams);

FrameKernelFn pick_kernel(int occ, int mode, int pair) {
  if (pair == 2) return mode == 0 ? conv_frame_kernel<1, 0, 2> : mode == 1 ? conv_frame_kernel<1, 1, 2> : conv_frame_kernel<1, 2, 2>;
  if (occ == 2) return mode == 0 ? conv_frame_kernel<2, 0, 1> : mode == 1 ? conv_frame_kernel<2, 1, 1> : conv_frame_kernel<2, 2, 1>;
  return mode == 0 ? conv_frame_kernel<1, 0, 1> : mode == 1 ? conv_frame_kernel<1, 1, 1> : conv_frame_kernel<1, 2, 1>;
}

int valid_taps(int o, int stride, int pad, int ks, int Hin) {
  int n = 0;
  for (int k = 0; k < ks; ++k) {
    const int i = o * stride + k - pad;
    n += (i >= 0 && i < Hin) ? 1 : 0;
  }
  return n;
}

}  // namespace

int conv_frame_plan(const ConvFrameProblem& pr, ConvFramePlan* plan) {
  AVH_CHECK(pr.A && pr.B && pr.C && pr.scale && pr.bias, "null pointer");
  AVH_CHECK(pr.Cin % 64 == 0 && pr.Cout % 64 == 0 && pr.Cout <= MAX_COUT, "unsupported channel count");
  AVH_CHECK((pr.ks == 3 || pr.ks == 1) && (pr.stride == 1 || pr.stride == 2), "unsupported kernel / stride");
  AVH_CHECK(pr.Hout >= 1 && pr.Hout <= 31 && pr.Sout >= pr.Hout && pr.Sin >= pr.Hin, "unsupported image size");
  AVH_CHECK(pr.frames >= 1 && pr.frames < 65535ll * BM, "frame count out of range");
  AVH_CHECK(pr.R == nullptr || pr.slope2 != nullptr, "residual form needs the second PReLU");
  plan->prob = pr;
  const int pad = pr.ks == 3 ? 1 : 0;
  int bn = pr.block_n, occ = pr.occ;
  if (bn == 0) bn = pr.Cout >= 256 ? 256 : pr.Cout;
  // CTA pairs (cta_group::2) for the 256-wide tiles of layers 3-4, single CTAs elsewhere.  Measured per step (2400
  // frames), pairs against single CTAs: 256-channel 3x3 convs 0.204 vs 0.232 ms, 512-channel 0.175 vs 0.179, but the
  // 128-channel layer (BN 128) 0.300 vs 0.284 ms against two single CTAs per SM.
  int pair = pr.pair != 0 ? pr.pair : (bn == 256 ? 2 : 1);
  if (device_sm_count() < 2 || bn % 128 != 0) pair = 1;        // each CTA of a pair stages bn / 2 weight rows (64-row boxes)
  if (pair == 2) occ = 1;
  if (occ == 0) occ = bn <= 128 ? 2 : 1;
  AVH_CHECK(bn % 64 == 0 && bn <= 256 && pr.Cout % bn == 0 && (occ == 1 || (occ == 2 && bn <= 128)), "bad tile shape");
  plan->prob.block_n = bn;
  plan->prob.occ = occ;
  plan->pair = pair;
  const int stage_bytes = A_STAGE_BYTES + (bn / pair) * BK * 2;
  const int smem_limit = occ == 2 ? FOcc<2>::SMEM_LIMIT : FOcc<1>::SMEM_LIMIT;
  const int epi_bytes = occ == 2 ? FOcc<2>::EPI_STAGE_BYTES : FOcc<1>::EPI_STAGE_BYTES;
  int stages = (smem_limit - 1024 - epi_bytes - COLVEC_BYTES - BAR_BYTES) / stage_bytes;
  if (stages > MAX_STAGES) stages = MAX_STAGES;
  AVH_CHECK(stages >= 2, "tile too large for shared memory");
  plan->stages = stages;
  plan->smem = 1024 + (size_t)stages * stage_bytes + epi_bytes + COLVEC_BYTES + BAR_BYTES;
  const long long a_cols = (long long)pr.Pin * pr.Cin, c_cols = (long long)pr.Pout * pr.Cout;
  AVH_CHECK(a_cols < (1ll << 31) && c_cols < (1ll << 31), "frame rows too wide");
  if (encode_2d(&plan->tma_a, pr.A, pr.frames, (int)a_cols, a_cols, BM)) return 1;
  const int b_cols = pr.ks * pr.ks * pr.Cin + (pr.A2 != nullptr ? pr.ds_Cin : 0);
  if (encode_2d(&plan->tma_b, pr.B, pr.Cout, b_cols, b_cols, bn / pair)) return 1;
  plan->tma_a2 = plan->tma_a;
  if (pr.A2 != nullptr) {
    AVH_CHECK(pr.ds_Cin % 64 == 0 && pr.ds_stride >= 1 && pr.ds_Sin >= 1, "bad shortcut geometry");
    const long long a2_cols = (long long)pr.ds_Pin * pr.ds_Cin;
    AVH_CHECK(a2_cols < (1ll << 31), "frame rows too wide");
    if (encode_2d(&plan->tma_a2, pr.A2, pr.frames, (int)a2_cols, a2_cols, BM)) return 1;
  }
  if (encode_c(&plan->tma_c, pr.C, pr.frames, (int)c_cols, c_cols, 0)) return 1;

  // ---- tile lists: longest-processing-time greedy over groups of frame blocks
  const int sms = device_sm_count();
  const int num_m = (int)((pr.frames + (long long)BM * pair - 1) / ((long long)BM * pair));   // frame blocks of a unit
  const int nsub = pr.Cout / bn;
  const int chunks = pr.Cin / 64;
  const long long tiles_total = (long long)num_m * pr.Hout * pr.Hout * nsub;
  const int grid = (int)std::min<long long>(tiles_total, (long long)sms * occ / pair);        // work units (CTAs or pairs)
  const double kblock = std::max(415.0, 2.0 * bn * occ);      // clk per k-block (gemm_tcgen05.cu model_cycles)
  const size_t in_frame_bytes = (size_t)a_cols * 2;
  int group = (int)std::max<size_t>(1, (size_t)(24u << 20) / (in_frame_bytes * BM * pair));
  struct T { int code; double cost; };
  std::vector<std::vector<int>> lists(grid);
  std::vector<double> load(grid, 0.0);
  for (int g0 = 0; g0 < num_m; g0 += group) {
    std::vector<T> ts;
    for (int m = g0; m < std::min(num_m, g0 + group); ++m)
      for (int oy = 0; oy < pr.Hout; ++oy)
        for (int ox = 0; ox < pr.Hout; ++ox) {
          const int nk = valid_taps(oy, pr.stride, pad, pr.ks, pr.Hin) * valid_taps(ox, pr.stride, pad, pr.ks, pr.Hin) * chunks +
                         (pr.A2 != nullptr ? pr.ds_Cin / 64 : 0);
          for (int s = 0; s < nsub; ++s)
            ts.push_back(T{m | (oy << 16) | (ox << 21) | (s << 26), nk * kblock + 500.0});
        }
    std::stable_sort(ts.begin(), ts.end(), [](const T& a, const T& b) { return a.cost > b.cost; });
    for (const T& t : ts) {
      int best = 0;
      for (int c = 1; c < grid; ++c)
        if (load[c] < load[best]) best = c;
      lists[best].push_back(t.code);
      load[best] += t.cost;
    }
  }
  std::vector<int> table(grid + 1);
  int off = grid + 1;
  for (int c = 0; c < grid; ++c) {
    table[c] = off;
    off += (int)lists[c].size();
  }
  table[grid] = off;
  for (int c = 0; c < grid; ++c) table.insert(table.end(), lists[c].begin(), lists[c].end());
  plan->grid = grid * pair;
  plan->tiles_host = table;
  return 0;
}

size_t conv_frame_table_bytes(const ConvFrameProblem& pr) {
  // upper bound usable before planning: one int per tile (narrowest tile) + offsets for 2 CTAs on each of <= 1024 SMs
  const long long num_m = (pr.frames + BM - 1) / BM;
  return (size_t)(num_m * pr.Hout * pr.Hout * (pr.Cout / 64) + 2 * 1024 + 1) * sizeof(int);
}

int conv_frame_bind_table(ConvFramePlan* plan, void* dev_table) {
  AVH_CUDA_OK(cudaMemcpy(dev_table, plan->tiles_host.data(), plan->tiles_host.size() * sizeof(int), cudaMemcpyHostToDevice));
  plan->tiles_dev = reinterpret_cast<const int*>(dev_table);
  return 0;
}

int conv_frame_launch(const ConvFramePlan& plan, cudaStream_t stream) {
  const ConvFrameProblem& pr = plan.prob;
  AVH_CHECK(plan.tiles_dev != nullptr, "tile table not bound");
  FrameParams p;
  p.frames = pr.frames;
  p.Hin = pr.Hin; p.Sin = pr.Sin; p.Cin = pr.Cin;
  p.Hout = pr.Hout; p.Sout = pr.Sout; p.Cout = pr.Cout;
  p.ks = pr.ks; p.stride = pr.stride; p.pad = pr.ks == 3 ? 1 : 0;
  p.block_n = pr.block_n; p.stages = plan.stages;
  p.chunks = pr.Cin / 64;
  p.ds_chunks = pr.A2 != nullptr ? pr.ds_Cin / 64 : 0;
  p.ds_stride = pr.ds_stride; p.ds_Sin = pr.ds_Sin; p.ds_Cin = pr.ds_Cin;
  p.ds_bcol = pr.ks * pr.ks * pr.Cin;
  p.ldr = (long long)pr.Pout * pr.Cout;
  p.tiles = plan.tiles_dev;
  p.scale = pr.scale; p.bias = pr.bias; p.slope1 = pr.slope1; p.slope2 = pr.slope2;
  p.R = reinterpret_cast<const __nv_bfloat16*>(pr.R);
  const int occ = pr.occ == 2 ? 2 : 1;
  const int mode = pr.R != nullptr ? 2 : (pr.slope1 != nullptr ? 1 : 0);
  FrameKernelFn fn = pick_kernel(occ, mode, plan.pair);
  if (ensure_dyn_smem(reinterpret_cast<const void*>(fn), occ == 2 ? FOcc<2>::SMEM_LIMIT : FOcc<1>::SMEM_LIMIT)) return 1;
  const int threads = occ == 2 ? FOcc<2>::NUM_THREADS : FOcc<1>::NUM_THREADS;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)plan.grid);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = plan.smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)plan.pair;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 2 : 1;
  AVH_CUDA_OK(cudaLaunchKernelEx(&cfg, fn, plan.tma_a, plan.tma_b, plan.tma_c, plan.tma_a2, p));
  count_launch(1);
  return 0;
}

}  // namespace avh
