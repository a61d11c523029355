// Multi-head self-attention on the 5th-generation tensor cores (tcgen05 / TMEM / TMA), head_dim 64, bf16 operands,
// fp32 scores / softmax statistics / output accumulation, key-padding mask as -inf.
//
// Replaces the attention core inside torch's F.multi_head_attention_forward as called by
// fairseq/fairseq/modules/multihead_attention.py:170-192 (baddbmm + softmax + bmm + the head-averaged [B,T,T]
// weights the encoder discards, wav2vec2.py:889).  Nothing of size T x T reaches global memory.
//
// One CTA = one (clip, head, tile of <= 128 query rows).  Input: the fused QKV projection [rows, 3*D] (q already
// scaled by head_dim^-0.5 at weight-fold time); output: the per-head context [rows, D].
//   warp 0      TMA producer: the Q tile, then key / value blocks through a ring of 128-byte-swizzled smem stages
//   warp 1      MMA issuer (one elected lane):
//                 S = Q K^T      tcgen05.mma, both operands K-major in smem, 128 x kv x 64 -> fp32 S in tensor memory
//                 O += P V       tcgen05.mma, A = P (bf16 pairs) read from TENSOR MEMORY, B = V in smem as it sits in
//                                global memory ([keys, 64 dims] = MN-major operand: no transpose anywhere)
//   warp 2      TMEM allocator
//   warps 4-7   softmax + epilogue, thread = query row (TMEM lane): tcgen05.ld of S, mask, row max, exp2, row sum,
//               P written back over S with tcgen05.st (bf16 pairs: 32 keys -> 16 columns), finally O / sum -> bf16
// Clips of up to 160 frames (the 6 s clip) take one key block: S is computed once and swept twice (max, then exp).
// Longer clips stream 128-key blocks twice: pass A computes the exact row maxima (S only, two S buffers so that the
// MMA of block j+1 overlaps the sweep of block j), pass B recomputes S, writes P = exp2(S - max) and accumulates O
// in tensor memory — no running-max rescaling of O, at the price of issuing the (cheap) QK^T MMAs twice.
// Two CTAs per SM (256 TMEM columns, <= 100 KB smem each) overlap one tile's MUFU-bound softmax with the other's
// loads and MMAs.
#include "common.cuh"
#include "gemm.h"
#include "kernels.h"

namespace avh {
namespace {

constexpr int HD = 64;
constexpr int QROWS = 128;                    // query rows per tile = TMEM lanes
constexpr int Q_BYTES = QROWS * HD * 2;       // 16 KB
constexpr int MAX_STAGES = 4;
constexpr int TMEM_COLS = 256;
constexpr int COL_O = 192;                    // fp32 O accumulator: columns [192, 256)
constexpr int COL_S1 = 128;                   // second S buffer (pass A only; O is not live then)
constexpr float LOG2E = 1.4426950408889634f;

struct AttnParams {
  const unsigned char* kpm;   // [B, T] key-padding mask or null
  __nv_bfloat16* out;         // [rows, D]
  const int* cu;              // [B + 1] first row of every clip (packed ragged batches) or null: clip b starts at b * T
  int T, D;
  int kv_rows;                // keys per block: round16(T) <= 160 (single block) or 128
  int stages, stage_bytes;
  int mask_floats;
};

__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// instruction descriptor with the B operand MN-major (bit 16): V sits in smem as [keys, dims]
__host__ __device__ constexpr uint32_t umma_idesc_bf16_bmn(int M, int N) { return umma_idesc_bf16(M, N) | (1u << 16); }

__global__ void __launch_bounds__(256, 2)
attention_tc_kernel(const __grid_constant__ CUtensorMap tma_q, const __grid_constant__ CUtensorMap tma_kv,
                    const AttnParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  uint8_t* sQ = smem;
  uint8_t* sKV = smem + Q_BYTES;
  float* sMask = reinterpret_cast<float*>(sKV + p.stages * p.stage_bytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(sMask) + p.mask_floats * 4);
  uint64_t* full_bar = bars;                    // [MAX_STAGES]
  uint64_t* empty_bar = bars + MAX_STAGES;      // [MAX_STAGES]
  uint64_t* bar_q = bars + 2 * MAX_STAGES;      // Q tile landed (TMA -> MMA)
  uint64_t* bar_s = bar_q + 1;                  // [2] S buffer ready (MMA -> softmax)
  uint64_t* bar_sfree = bar_s + 2;              // [2] S buffer consumed (softmax -> MMA), pass A
  uint64_t* bar_p = bar_sfree + 2;              // P written (softmax -> MMA)
  uint64_t* bar_o = bar_p + 1;                  // O complete (MMA -> epilogue)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_o + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.z, h = blockIdx.y;
  pdl_launch_dependents();
  // clip geometry (cu_rows are written by the host before the forward: launch constants)
  const int row_base = p.cu != nullptr ? __ldg(p.cu + b) : b * p.T;
  const int Tb = p.cu != nullptr ? __ldg(p.cu + b + 1) - row_base : p.T;
  const int ntiles = (Tb + QROWS - 1) / QROWS;
  if ((int)blockIdx.x >= ntiles) return;            // clips shorter than the longest have fewer query tiles
  const int tile_rows = (Tb + ntiles - 1) / ntiles;         // balanced tiles: 150 frames -> 75 + 75
  const int kv = p.kv_rows;
  const int nkb = (Tb + kv - 1) / kv;
  const bool two_pass = nkb > 1;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_q);
    tma_prefetch_desc(&tma_kv);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < MAX_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(bar_q, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&bar_s[s], 1);
      mbar_init(&bar_sfree[s], 4);
    }
    mbar_init(bar_p, 4);
    mbar_init(bar_o, 1);
    mbar_fence_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    const int col_q = h * HD, col_k = p.D + h * HD, col_v = 2 * p.D + h * HD;
    int stage = 0;
    uint32_t phase = 0;
    if (elect_one()) {
      mbar_expect_tx(bar_q, Q_BYTES);
      tma_load_2d(sQ, &tma_q, bar_q, col_q, row_base + (int)blockIdx.x * tile_rows);
    }
    __syncwarp();
    const int nloads = two_pass ? 3 * nkb : 2;
    for (int i = 0; i < nloads; ++i) {
      // order of use: pass A K_0..K_{n-1}; pass B K_0, V_0, K_1, V_1, ...
      int blk, col;
      if (two_pass && i < nkb) { blk = i; col = col_k; }
      else {
        const int j = two_pass ? i - nkb : i;
        blk = j >> 1;
        col = (j & 1) ? col_v : col_k;
      }
      mbar_wait(&empty_bar[stage], phase ^ 1);
      if (elect_one()) {
        mbar_expect_tx(&full_bar[stage], (uint32_t)p.stage_bytes);
        tma_load_2d(sKV + stage * p.stage_bytes, &tma_kv, &full_bar[stage], col, row_base + blk * kv);
      }
      __syncwarp();
      if (++stage == p.stages) { stage = 0; phase ^= 1; }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    const uint32_t idesc_s = umma_idesc_bf16(QROWS, kv);
    const uint32_t idesc_o = umma_idesc_bf16_bmn(QROWS, HD);
    int stage = 0;
    uint32_t phase = 0;
    const uint64_t qdesc = umma_desc_sw128(smem_u32(sQ));
    uint32_t sfree_phase[2] = {0, 0};
    uint32_t p_phase = 0;
    mbar_wait(bar_q, 0);
    tc_fence_after();
    if (two_pass) {
      for (int j = 0; j < nkb; ++j) {
        const int buf = j & 1;
        if (j >= 2) {              // the sweep of the S that lived in this buffer two blocks ago is done
          mbar_wait(&bar_sfree[buf], sfree_phase[buf]);
          sfree_phase[buf] ^= 1;
          tc_fence_after();
        }
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint64_t kdesc = umma_desc_sw128(smem_u32(sKV + stage * p.stage_bytes));
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < HD / 16; ++k)
            umma_bf16(tmem_base + (buf ? COL_S1 : 0), qdesc + 2 * k, kdesc + 2 * k, idesc_s, k != 0);
          umma_commit(&empty_bar[stage]);
          umma_commit(&bar_s[buf]);
        }
        __syncwarp();
        if (++stage == p.stages) { stage = 0; phase ^= 1; }
      }
      // pass B writes S into buffer 0 and O over buffer 1: the last sweep of either buffer must have drained
      for (int buf = 0; buf < 2; ++buf) {
        mbar_wait(&bar_sfree[buf], sfree_phase[buf]);
        sfree_phase[buf] ^= 1;
      }
      tc_fence_after();
    }
    for (int j = 0; j < nkb; ++j) {
      // S_j = Q K_j^T into buffer 0 (in-order execution behind PV_{j-1}, which reads P from the same columns)
      mbar_wait(&full_bar[stage], phase);
      tc_fence_after();
      const uint64_t kdesc = umma_desc_sw128(smem_u32(sKV + stage * p.stage_bytes));
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < HD / 16; ++k) umma_bf16(tmem_base, qdesc + 2 * k, kdesc + 2 * k, idesc_s, k != 0);
        if (two_pass) umma_commit(&empty_bar[stage]);      // a single key block is loaded once: no stage is reused
        umma_commit(&bar_s[0]);
      }
      __syncwarp();
      if (++stage == p.stages) { stage = 0; phase ^= 1; }
      // O += P_j V_j
      mbar_wait(bar_p, p_phase);
      p_phase ^= 1;
      mbar_wait(&full_bar[stage], phase);
      tc_fence_after();
      const uint64_t vdesc = umma_desc_sw128(smem_u32(sKV + stage * p.stage_bytes));
      const int ksteps = (min(kv, Tb - j * kv) + 15) >> 4;    // 16 keys per MMA; keys past the clip have P = 0
      if (elect_one()) {
        for (int k = 0; k < ksteps; ++k)
          umma_bf16_ts(tmem_base + COL_O, tmem_base + 8 * k, vdesc + 128 * k, idesc_o, (j | k) != 0);
        if (two_pass) umma_commit(&empty_bar[stage]);
        if (j + 1 == nkb) umma_commit(bar_o);
      }
      __syncwarp();
      if (++stage == p.stages) { stage = 0; phase ^= 1; }
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ softmax + epilogue: thread = query row
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;                 // row inside the tile = TMEM lane
    const uint32_t lane_addr = tmem_base + ((uint32_t)(quarter * 32) << 16);
    // additive key mask: 0 for live keys, -inf for padded keys and keys past the clip
    for (int k = threadIdx.x - 128; k < nkb * kv; k += 128) {
      const bool dead = k >= Tb || (p.kpm != nullptr && p.kpm[(long long)b * p.T + k] != 0);
      sMask[k] = dead ? -INFINITY : 0.f;
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");
    const int nchunks = kv >> 5;                         // 32-key chunks per block (kv is a multiple of 32)
    uint32_t s_phase[2] = {0, 0};
    const int q0 = (int)blockIdx.x * tile_rows;
    const int q_valid = min(tile_rows, Tb - q0);
    const bool warp_live = quarter * 32 < q_valid;     // warps whose 32 rows are all past the tile skip the math
    float m = -INFINITY;
    if (two_pass) {
      for (int j = 0; j < nkb; ++j) {
        const int buf = j & 1;
        mbar_wait(&bar_s[buf], s_phase[buf]);
        s_phase[buf] ^= 1;
        tc_fence_after();
        if (warp_live) {
          const int nch = (min(kv, Tb - j * kv) + 31) >> 5;
          for (int c = 0; c < nch; ++c) {
            uint32_t v[32];
            tmem_ld_32x32(lane_addr + (buf ? COL_S1 : 0) + 32 * c, v);
            tmem_ld_wait();
            const float* mk = sMask + j * kv + 32 * c;
#pragma unroll
            for (int i = 0; i < 32; ++i) m = fmaxf(m, __uint_as_float(v[i]) + mk[i]);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar_sfree[buf]);
      }
    }
    float l = 0.f;
    for (int j = 0; j < nkb; ++j) {
      mbar_wait(&bar_s[0], s_phase[0]);
      s_phase[0] ^= 1;
      tc_fence_after();
      if (warp_live) {
        const int nch = two_pass ? (min(kv, Tb - j * kv) + 31) >> 5 : nchunks;
        const float* mk0 = sMask + j * kv;
        if (!two_pass) {
          for (int c = 0; c < nch; ++c) {
            uint32_t v[32];
            tmem_ld_32x32(lane_addr + 32 * c, v);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) m = fmaxf(m, __uint_as_float(v[i]) + mk0[32 * c + i]);
          }
        }
        const float ms = (m == -INFINITY) ? 0.f : m * LOG2E;      // fully masked row: every p = exp2(-inf) = 0
        for (int c = 0; c < nch; ++c) {
          uint32_t v[32];
          tmem_ld_32x32(lane_addr + 32 * c, v);
          tmem_ld_wait();
          uint32_t pk[16];
          const float* mk = mk0 + 32 * c;
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const float p0 = ex2(fmaf(__uint_as_float(v[2 * i]) + mk[2 * i], LOG2E, -ms));
            const float p1 = ex2(fmaf(__uint_as_float(v[2 * i + 1]) + mk[2 * i + 1], LOG2E, -ms));
            l += p0 + p1;
            pk[i] = pack_bf16(p0, p1);
          }
          tmem_st_32x16(lane_addr + 16 * c, pk);      // P chunk c over S columns already consumed
        }
        tmem_st_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_p);
    }
    // ---- epilogue: O / l -> bf16 -> global (128 B per row)
    mbar_wait(bar_o, 0);
    tc_fence_after();
    uint32_t o0[32], o1[32];
    if (warp_live) {
      tmem_ld_32x32(lane_addr + COL_O, o0);
      tmem_ld_32x32(lane_addr + COL_O + 32, o1);
      tmem_ld_wait();
    }
    if (warp_live && row < q_valid) {
      const float inv = l > 0.f ? 1.f / l : 0.f;
      uint4* dst = reinterpret_cast<uint4*>(p.out + (long long)(row_base + q0 + row) * p.D + h * HD);
#pragma unroll
      for (int i = 0; i < 4; ++i)
        dst[i] = make_uint4(pack_bf16(__uint_as_float(o0[8 * i]) * inv, __uint_as_float(o0[8 * i + 1]) * inv),
                            pack_bf16(__uint_as_float(o0[8 * i + 2]) * inv, __uint_as_float(o0[8 * i + 3]) * inv),
                            pack_bf16(__uint_as_float(o0[8 * i + 4]) * inv, __uint_as_float(o0[8 * i + 5]) * inv),
                            pack_bf16(__uint_as_float(o0[8 * i + 6]) * inv, __uint_as_float(o0[8 * i + 7]) * inv));
#pragma unroll
      for (int i = 0; i < 4; ++i)
        dst[4 + i] = make_uint4(pack_bf16(__uint_as_float(o1[8 * i]) * inv, __uint_as_float(o1[8 * i + 1]) * inv),
                                pack_bf16(__uint_as_float(o1[8 * i + 2]) * inv, __uint_as_float(o1[8 * i + 3]) * inv),
                                pack_bf16(__uint_as_float(o1[8 * i + 4]) * inv, __uint_as_float(o1[8 * i + 5]) * inv),
                                pack_bf16(__uint_as_float(o1[8 * i + 6]) * inv, __uint_as_float(o1[8 * i + 7]) * inv));
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 2) tmem_dealloc(tmem_base, TMEM_COLS);
}

}  // namespace

// tensor maps over the QKV matrix (built once per plan) + launch geometry
int attention_tc_plan(const void* qkv, long long rows, int B, int T, int D, int H, AttnTcPlan* plan) {
  AVH_CHECK(D == H * HD, "attention kernel requires head_dim 64");
  AVH_CHECK(T >= 1 && B >= 1, "empty attention problem");
  plan->B = B; plan->T = T; plan->D = D; plan->H = H;
  plan->kv_rows = T <= 160 ? ((T + 31) / 32) * 32 : 128;      // whole 32-key chunks (sweeps) and 16-key MMAs
  plan->stages = T <= 160 ? 2 : MAX_STAGES;
  plan->stage_bytes = plan->kv_rows * HD * 2;
  const int nkb = (T + plan->kv_rows - 1) / plan->kv_rows;
  plan->mask_floats = nkb * plan->kv_rows;
  plan->smem = 1024 + Q_BYTES + (size_t)plan->stages * plan->stage_bytes + (size_t)plan->mask_floats * 4 + 256;      // 15 mbarriers + TMEM slot
  AVH_CHECK(plan->smem <= 113 * 1024, "clip too long for the attention kernel's key-mask buffer");
  if (encode_2d(&plan->tma_q, qkv, rows, 3 * D, 3ll * D, QROWS)) return 1;
  if (encode_2d(&plan->tma_kv, qkv, rows, 3 * D, 3ll * D, plan->kv_rows)) return 1;
  return 0;
}

int attention_tc_launch(const AttnTcPlan& plan, const unsigned char* kpm, const int* cu, void* out, cudaStream_t stream) {
  AttnParams p;
  p.kpm = kpm;
  p.out = reinterpret_cast<__nv_bfloat16*>(out);
  p.cu = cu;
  p.T = plan.T; p.D = plan.D;
  p.kv_rows = plan.kv_rows;
  p.stages = plan.stages; p.stage_bytes = plan.stage_bytes;
  p.mask_floats = plan.mask_floats;
  if (ensure_dyn_smem(reinterpret_cast<const void*>(attention_tc_kernel), 113 * 1024)) return 1;
  // One query tile per CTA.  Several consecutive tiles of a head per CTA (K/V loaded once, 256 CTAs = one wave at
  // T = 150) measured slower or no better: 11.4 vs 11.7 us at 16 x 150 and 38 vs 32 us at 4 x 600; the tiles of a CTA
  // run back to back, so the softmax of one cannot overlap the MMAs of the next.
  const int ntiles = (plan.T + QROWS - 1) / QROWS;
  dim3 grid(ntiles, plan.H, plan.B);
  AVH_CUDA_OK(launch_pdl(attention_tc_kernel, grid, dim3(256), plan.smem, stream, plan.tma_q, plan.tma_kv, p));
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

}  // namespace avh
