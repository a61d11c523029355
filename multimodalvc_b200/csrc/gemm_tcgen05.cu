// tcgen05 / TMEM / TMA GEMM for sm_100a (B200): C[M,N] = epilogue(A[M,K] * B[N,K]^T), bf16 in, fp32 accumulate.
//
// Persistent and warp-specialised.  Work unit: a (PAIR*128) x BN output tile owned by a cluster of PAIR CTAs
// (PAIR = 1: single-CTA 128 x BN tiles, the default; PAIR = 2: one CTA pair on the two SMs of a TPC drives ONE
// tcgen05.mma.cta_group::2 of shape 256 x BN x 16, each CTA staging its own 128 rows of A and HALF of B).
//   warp 0      TMA producer (one lane): A/B k-blocks into a ring of 128-byte-swizzled K-major smem stages,
//               out-of-bounds rows/columns zero-filled by TMA
//   warp 1      MMA issuer (one lane, leader CTA only): tcgen05.mma into TMEM, two accumulator stages of 256
//               columns so the epilogue of tile i overlaps the main loop of tile i+1; tcgen05.commit (multicast
//               to both CTAs in pair mode) frees smem stages and publishes finished accumulators
//   warp 2      TMEM allocator
//   warps 4-11  epilogue.  Fast path, thread = row: tcgen05.ld -> fused per-column scale/bias, PReLU /
//               erf-GELU, residual add, second PReLU, row masking -> 128-byte-swizzled smem box -> TMA store,
//               or TMA reduce-add straight into the fp32 residual stream (x += acc + bias without loading x).
//               Re-mapped outputs (stride-2 conv rows, positional conv) take a per-thread path that transposes
//               32x32 chunks through smem so that global accesses are row-contiguous.
// BN is a run-time multiple of 32 (<= 256) chosen per problem by a measured cost model (whole waves over the
// 148 SMs; one k-block costs ~max(4*55, 2*BN) + 170 clk).  The K loop walks a table of
// (A column, A row shift, B column) steps, so the same kernel runs plain Linear layers, shifted-row
// implicit-GEMM convolutions (3x3 trunk convs, the 5 temporal taps of the stem, the 128 taps of the grouped
// positional conv) and split-precision (bf16 hi/mid plane) fp32-faithful products.  The epilogue variant is a
// template parameter: predicated-off options are not free in the 8 epilogue warps (the fully dynamic form
// issues ~1500 instructions per 32x32 chunk) and the epilogue is what bounds short-K GEMMs.
//
// Replaces on the reference path (all cuBLAS/cuDNN library calls there): nn.Linear in
// avhubert/hubert.py:321,360-364, fairseq/fairseq/models/wav2vec/wav2vec2.py:955-956,
// multihead_attention.py:64-77; nn.Conv1d pos_conv wav2vec2.py:822-835; nn.Conv2d / Conv3d avhubert/resnet.py:15-24,138.
#include "common.cuh"
#include "gemm.h"

#include <cstdlib>
#include <mutex>
#include <set>

namespace avh {

namespace {

constexpr int BM = 128;                       // rows per CTA
constexpr int BK = 64;                        // K elements per stage (one 128-byte swizzle row)
constexpr int A_STAGE_BYTES = BM * BK * 2;    // 16 KB
constexpr int MAX_STAGES = 8;
constexpr int COLVEC_BYTES = 2 * 4 * 256 * 4;              // per-tile bias/scale/slope vectors, double-buffered (8 KB)
constexpr int BAR_BYTES = (2 * MAX_STAGES + 4) * 8 + 16;

// OCC = CTAs resident per SM.  OCC 1: 8 epilogue warps, all 512 TMEM columns (BN <= 256), 227 KB of smem.
// OCC 2: two independent CTAs per SM, each with its own TMA producer and MMA-issuing thread, 4 epilogue warps,
// 256 TMEM columns (BN <= 128) and <= 113 KB of smem.  One elected lane sustains one tcgen05.mma per ~53 clk
// (tools/micro/mma_bench.cu), i.e. it saturates the tensor pipe for N >= 128 but only 59 % of it for N = 64:
// narrow tiles (stem, layer1 convolutions) want two issuers per SM.
template <int OCC>
struct Occ {
  static constexpr int EPI_WARPS = OCC == 2 ? 4 : 8;
  static constexpr int NUM_THREADS = 128 + 32 * EPI_WARPS;    // producer, mma, alloc, spare + epilogue warps
  static constexpr int TMEM_COLS = 512 / OCC;
  static constexpr int ACC_STRIDE = 256 / OCC;                // TMEM columns per accumulator stage
  static constexpr int EPI_STAGE_BYTES = EPI_WARPS * 4096;    // per-warp 32 rows x 128 B staging boxes.  (Two boxes per warp,
                                                              // so that the store of box i drains under box i+1, cost a pipeline
                                                              // stage: fc1 20.6 -> 23.3 us, fc2 23.0 -> 25.1 us, qkv unchanged.)
  static constexpr int SMEM_LIMIT = OCC == 2 ? 113 * 1024 : 227 * 1024;
  static constexpr int HSTRIDE = EPI_WARPS / 4;               // column-box interleave between epilogue warp sets
};

struct KernelParams {
  long long M;
  int N;
  int num_kb;
  int num_m_blk, num_n_blk;     // m blocks in units of PAIR*128 rows
  int block_n;
  int stages;
  int ktab_bytes;               // smem reserved for the K-step table (multiple of 1024; 0 without a table)
  int a_col_per_nblk;
  const int* a_col_nblk;
  const int4* ktable;
  int c_mode;                   // 0 = per-thread global stores, 1 = TMA store of C, 2 = TMA reduce-add into C (= R)
  unsigned long long* trace;    // debug: [grid][16] SM clock stamps (null in production)
  // stream-K (sk != 0): the tile x k-block space is cut into one contiguous range per work unit; a unit whose range
  // starts inside a tile writes that partial accumulator (fp32) to sk_ws[unit] and raises sk_flags[unit]; the unit that
  // holds the tile's first k-block owns the tile: it adds the partials of the following units in unit order (fixed
  // partition + fixed order = bit-identical reruns) and runs the epilogue.  Flags are reset by their consumer.
  int sk;
  float* sk_ws;                 // [units][PAIR * 128][block_n] fp32
  int* sk_flags;                // [units], zero between launches
  Epilogue ep;
};

// debug stall accounting (only when a trace buffer is attached): cycles a role spent blocked on an mbarrier
#ifdef AVH_STALL_ACC
#define AVH_WAIT_ACC(bar, parity, acc)                    \
  do {                                                    \
    if (p.trace == nullptr) mbar_wait((bar), (parity));   \
    else {                                                \
      const long long _c0 = clock64();                    \
      mbar_wait((bar), (parity));                         \
      (acc) += clock64() - _c0;                           \
    }                                                     \
  } while (0)
#else
// production build: a plain wait (the run-time test sat between the MMAs of the issue loop: tools/ab_bench.sh)
#define AVH_WAIT_ACC(bar, parity, acc) \
  do {                                 \
    mbar_wait((bar), (parity));        \
    (void)(acc);                       \
  } while (0)
#endif

#define AVH_TRACE(slot)                                                                            \
  do {                                                                                             \
    if (p.trace != nullptr) p.trace[(size_t)blockIdx.x * 16 + (slot)] = (unsigned long long)clock64(); \
  } while (0)

// Work of one unit (CTA or CTA pair): classic persistent tiles (tile = unit, unit + units, ...; whole K each) or, in
// stream-K mode, the k-blocks [unit * U / units, (unit + 1) * U / units) of the tile-major k-block sequence.
struct SegIter {
  int sk, num_kb, num_units;
  int tile, tiles_end;          // persistent mode
  long long pos, end;           // stream-K mode
  __device__ __forceinline__ SegIter(int sk_, int unit, int num_units_, int num_tiles, int num_kb_)
      : sk(sk_), num_kb(num_kb_), num_units(num_units_), tile(unit), tiles_end(num_tiles) {
    const long long U = (long long)num_tiles * num_kb_;
    pos = (long long)unit * U / num_units_;
    end = (long long)(unit + 1) * U / num_units_;
  }
  // next segment: tile index and k-block range [kb0, kb1); false when the unit's work is done
  __device__ __forceinline__ bool next(int& t, int& kb0, int& kb1) {
    if (!sk) {
      if (tile >= tiles_end) return false;
      t = tile; kb0 = 0; kb1 = num_kb;
      tile += num_units;
      return true;
    }
    if (pos >= end) return false;
    t = (int)(pos / num_kb);
    kb0 = (int)(pos - (long long)t * num_kb);
    const long long left = end - pos;
    kb1 = left < (long long)(num_kb - kb0) ? kb0 + (int)left : num_kb;
    pos += kb1 - kb0;
    return true;
  }
};

// ACT (ACT_*), RES (residual add), S2 (second PReLU), SCALE (per-column scale) and OUTF32 (fp32 output and
// residual, else bf16) are compile-time when >= 0 and read from the Epilogue struct when -1.
// SK: stream-K code compiled in (only the instantiations the planner picks for a stream-K launch carry it: with the
// code in every kernel the epilogue spilled registers and the encoder GEMMs ran ~9 % slower — tools/ab_bench.sh).
template <int PAIR, int OCC, int ACT, int RES, int S2, int SCALE, int OUTF32, int SK = 0>
__global__ void __launch_bounds__(Occ<OCC>::NUM_THREADS, OCC)
gemm_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
            const __grid_constant__ CUtensorMap tma_c, const KernelParams p) {
  constexpr int EPI_WARPS = Occ<OCC>::EPI_WARPS;
  constexpr int NUM_THREADS = Occ<OCC>::NUM_THREADS;
  constexpr int TMEM_COLS = Occ<OCC>::TMEM_COLS;
  constexpr int ACC_STRIDE = Occ<OCC>::ACC_STRIDE;
  constexpr int EPI_STAGE_BYTES = Occ<OCC>::EPI_STAGE_BYTES;
  constexpr int HSTRIDE = Occ<OCC>::HSTRIDE;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  const int BN = p.block_n;
  const int STAGES = p.stages;
  const int b_stage_bytes = (BN / PAIR) * BK * 2;
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + STAGES * A_STAGE_BYTES;
  uint8_t* epi_stage = smem_b + STAGES * b_stage_bytes;
  float* colvec = reinterpret_cast<float*>(epi_stage + EPI_STAGE_BYTES);
  int4* ktab = reinterpret_cast<int4*>(reinterpret_cast<uint8_t*>(colvec) + COLVEC_BYTES);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(ktab) + p.ktab_bytes);
  uint64_t* empty_bar = full_bar + MAX_STAGES;
  uint64_t* tmem_full = empty_bar + MAX_STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int cta_rank = PAIR == 2 ? (int)cluster_ctarank() : 0;
  const bool leader = cta_rank == 0;
  const int unit = blockIdx.x / PAIR;                 // cluster index
  const int num_units = gridDim.x / PAIR;
  const int num_tiles = p.num_m_blk * p.num_n_blk;
  pdl_launch_dependents();            // the next kernel of the stream may start its own prologue
  if (threadIdx.x == 0) AVH_TRACE(0);

  if (p.ktable != nullptr) {
    for (int i = threadIdx.x; i < p.num_kb; i += NUM_THREADS) ktab[i] = __ldg(p.ktable + i);
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
    if (p.c_mode != 0) tma_prefetch_desc(&tma_c);
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
  // Weights are launch constants too: the B tiles of the first pipeline stages go in flight BEFORE the dependency
  // wait (they come from DRAM — 25 MB of weights per layer never stay in L2 — and were the longest part of the
  // 1.1 us between the wait and the first MMA); the A tiles (activations) follow after the wait.
  int pre_b = 0;
  if (PAIR == 1 && warp == 0) {
    SegIter first(SK != 0 ? p.sk : 0, unit, num_units, num_tiles, p.num_kb);
    int t0, f_kb0 = 0, f_kb1 = 0;
    if (first.next(t0, f_kb0, f_kb1)) {
    const int n_blk0 = t0 / p.num_m_blk;
    pre_b = f_kb1 - f_kb0 < STAGES ? f_kb1 - f_kb0 : STAGES;
    const uint32_t stage_tx0 = (uint32_t)(A_STAGE_BYTES + b_stage_bytes);
    for (int kb = 0; kb < pre_b; ++kb) {
      int4 e;
      if (p.ktable != nullptr) e = ktab[f_kb0 + kb];
      else e = make_int4((f_kb0 + kb) * BK, 0, (f_kb0 + kb) * BK, 0);
      if (elect_one()) {
        mbar_expect_tx(&full_bar[kb], stage_tx0);
        tma_load_2d(smem_b + kb * b_stage_bytes, &tma_b, &full_bar[kb], e.z, n_blk0 * BN + e.w);
      }
      __syncwarp();
    }
    }
  }
  // everything above (K table, barrier init, TMEM allocation, descriptor prefetch, first weight tiles) touched only
  // launch-constant data; from here on the kernel reads and writes activations of its predecessors
  pdl_wait();
  if (threadIdx.x == 0) AVH_TRACE(1);

  // Producer and MMA warps run their loops with ALL lanes (warp-uniform operands stay in uniform registers) and
  // elect one lane only for the issue itself.  A loop entered by a single lane makes the compiler wrap every
  // UTCHMMA / UTMALDG in an ELECT/BRA.U.ANY "uniformisation" loop: ~105 clk per tcgen05.mma instead of ~53
  // (tools/micro/mma_bench.cu modes 0 vs 6), which capped every tile narrower than 256 columns.
  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (both CTAs)
    int stage = 0;
    uint32_t phase = 0;
    long long prod_wait = 0;
    const uint32_t stage_tx = (uint32_t)PAIR * (uint32_t)(A_STAGE_BYTES + b_stage_bytes);
    SegIter segs(SK != 0 ? p.sk : 0, unit, num_units, num_tiles, p.num_kb);
    int tile, kb0, kb1;
    bool first_seg = true;
    for (; segs.next(tile, kb0, kb1); first_seg = false) {
      const int m_blk = tile % p.num_m_blk;
      const int n_blk = tile / p.num_m_blk;
      const int m0 = (m_blk * PAIR + cta_rank) * BM;
      const int n0 = n_blk * BN + cta_rank * (BN / PAIR);
      const int a_col_base = p.a_col_nblk != nullptr ? __ldg(p.a_col_nblk + n_blk) : n_blk * p.a_col_per_nblk;
      for (int kb = kb0; kb < kb1; ++kb) {
        int4 e;
        if (p.ktable != nullptr) e = ktab[kb];
        else e = make_int4(kb * BK, 0, kb * BK, 0);
        AVH_WAIT_ACC(&empty_bar[stage], phase ^ 1, prod_wait);
        const bool b_early = PAIR == 1 && first_seg && kb - kb0 < pre_b;   // B tile already requested before the wait
        if (elect_one()) {
          if (leader && !b_early) mbar_expect_tx(&full_bar[stage], stage_tx);
          if (PAIR == 2) {
            tma_load_2d_pair(smem_a + stage * A_STAGE_BYTES, &tma_a, &full_bar[stage], e.x + a_col_base, m0 + e.y);
            tma_load_2d_pair(smem_b + stage * b_stage_bytes, &tma_b, &full_bar[stage], e.z, n0 + e.w);
          } else {
            tma_load_2d(smem_a + stage * A_STAGE_BYTES, &tma_a, &full_bar[stage], e.x + a_col_base, m0 + e.y);
            if (!b_early) tma_load_2d(smem_b + stage * b_stage_bytes, &tma_b, &full_bar[stage], e.z, n0 + e.w);
          }
          if (first_seg && kb == kb0) AVH_TRACE(2);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
    if (p.trace != nullptr && lane == 0) p.trace[(size_t)blockIdx.x * 16 + 14] = (unsigned long long)prod_wait;
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA only)
    if (leader) {
      const uint32_t idesc = umma_idesc_bf16(BM * PAIR, BN);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      long long wait_full = 0, wait_tmem = 0;
      SegIter segs(SK != 0 ? p.sk : 0, unit, num_units, num_tiles, p.num_kb);
      int tile, kb0, kb1;
      for (; segs.next(tile, kb0, kb1); ++it) {
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        AVH_WAIT_ACC(&tmem_empty[acc], acc_phase ^ 1, wait_tmem);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * ACC_STRIDE;
        for (int kb = kb0; kb < kb1; ++kb) {
          AVH_WAIT_ACC(&full_bar[stage], phase, wait_full);
          tc_fence_after();
          const uint64_t adesc = umma_desc_sw128(smem_u32(smem_a + stage * A_STAGE_BYTES));
          const uint64_t bdesc = umma_desc_sw128(smem_u32(smem_b + stage * b_stage_bytes));
          if (elect_one()) {
            if (it == 0 && kb == kb0) AVH_TRACE(3);
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) {
              // advance 16 bf16 (32 B) along K inside the 128-byte swizzle atom: +2 in 16-byte units
              if (PAIR == 2) umma_bf16_pair(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb > kb0) || (k != 0));
              else umma_bf16(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb > kb0) || (k != 0));
            }
            if (PAIR == 2) umma_commit_pair(&empty_bar[stage]);   // smem slot reusable in BOTH CTAs
            else umma_commit(&empty_bar[stage]);
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        if (elect_one()) {
          if (PAIR == 2) umma_commit_pair(&tmem_full[acc]);        // accumulator complete -> both epilogues
          else umma_commit(&tmem_full[acc]);
          if (it == 0) AVH_TRACE(4);
          AVH_TRACE(5);
        }
        __syncwarp();
      }
      if (p.trace != nullptr && lane == 0) {
        p.trace[(size_t)blockIdx.x * 16 + 12] = (unsigned long long)wait_full;
        p.trace[(size_t)blockIdx.x * 16 + 13] = (unsigned long long)wait_tmem;
      }
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ epilogue (both CTAs)
    const Epilogue& ep = p.ep;
    const int q = warp & 3;               // TMEM lane quarter this warp may access
    const int half = (warp - 4) >> 2;     // which interleaved set of column boxes this warp handles
    const int act = ACT >= 0 ? ACT : ep.act;
    const bool has_s2 = S2 >= 0 ? S2 != 0 : ep.slope2 != nullptr;
    const bool has_scale = SCALE >= 0 ? SCALE != 0 : ep.col_scale != nullptr;
    const bool out_f32 = OUTF32 >= 0 ? OUTF32 != 0 : ep.c_fp32 != 0;
    const bool res_any = RES >= 0 ? RES != 0 : ep.R != nullptr;
    int it = 0;
    SegIter segs(SK != 0 ? p.sk : 0, unit, num_units, num_tiles, p.num_kb);
    int tile, kb0, kb1;
    for (; segs.next(tile, kb0, kb1); ++it) {
      const int m_blk = tile % p.num_m_blk;
      const int n_blk = tile / p.num_m_blk;
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int row0 = (m_blk * PAIR + cta_rank) * BM + q * 32;     // first row of this warp's quarter
      if (SK != 0 && p.sk && kb0 > 0) {
        // ---- stream-K, tail part of a tile owned by an earlier unit: raw fp32 accumulator -> workspace slot of this
        //      unit (thread = row, 128 contiguous bytes per 32-column chunk), then raise the flag
        mbar_wait(&tmem_full[acc], acc_phase);
        tc_fence_after();
        // slot layout: float4 index ((chunk * 8 + j) * 128 + row): the 32 lanes of a warp write (and the owner reads)
        // 512 contiguous bytes per instruction — the row-major form (32 cache lines per instruction) cost 11 us per GEMM
        uint4* wslot = reinterpret_cast<uint4*>(p.sk_ws + ((size_t)unit * PAIR + cta_rank) * (size_t)BM * BN) + q * 32 + lane;
        const uint32_t taddr_p = tmem_base + ((uint32_t)(q * 32) << 16) + acc * ACC_STRIDE;
        for (int ch = half; ch < BN / 32; ch += HSTRIDE) {
          uint32_t rawv[32];
          tmem_ld_32x32(taddr_p + ch * 32, rawv);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 8; ++j)
            wslot[(size_t)(ch * 8 + j) * BM] = make_uint4(rawv[4 * j], rawv[4 * j + 1], rawv[4 * j + 2], rawv[4 * j + 3]);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (PAIR == 2) mbar_arrive_leader(&tmem_empty[acc]);
          else mbar_arrive(&tmem_empty[acc]);
        }
        __threadfence();
        asm volatile("bar.sync 1, %0;" ::"n"(32 * EPI_WARPS) : "memory");
        // one flag per CTA of the unit: the consumer CTA of the same rank reads exactly the rows this CTA wrote
        if (threadIdx.x == 128) atomicExch(p.sk_flags + unit * PAIR + cta_rank, 1);
        continue;
      }
      // stream-K owner of a tile whose K range continues in the following units: their partials are added (in unit
      // order) to the accumulator values before the epilogue math
      int sk_first = 0, sk_last = -1;
      if (SK != 0 && p.sk && kb1 < p.num_kb) {
        const long long U = (long long)num_tiles * p.num_kb;
        const long long tile_end = (long long)(tile + 1) * p.num_kb;
        sk_first = unit + 1;
        sk_last = unit + 1;
        while ((long long)(sk_last + 1) * U / num_units < tile_end) ++sk_last;     // unit whose range reaches the tile end
        if (lane == 0) {
          for (int v = sk_first; v <= sk_last; ++v) {
            const uint64_t t0w = global_timer_ns();
            while (*reinterpret_cast<volatile int*>(p.sk_flags + v * PAIR + cta_rank) == 0) {
              if (global_timer_ns() - t0w > 4000000000ull) { printf("avh: stream-K flag watchdog unit=%d waits %d\n", unit, v); __trap(); }
            }
          }
          __threadfence();
        }
        __syncwarp();
      }
      const long long r = (long long)row0 + lane;
      bool store = r < p.M;
      bool zero = false;
      long long orow = r;
      if (ep.map_mode == MAP_2LEVEL) {
        const long long n = r / ep.S2;
        const int rem = (int)(r - n * ep.S2);
        const int h = rem / ep.S1;
        const int w = rem - h * ep.S1;
        orow = n * ep.O2 + (long long)h * ep.O1 + w + ep.O0;
        if (!(h < ep.H && w < ep.W)) {
          if (ep.invalid_zero) zero = true; else store = false;
        }
      }
      if (ep.row_map != nullptr) {
        const int mr = r < p.M ? __ldg(ep.row_map + r) : -1;
        orow = mr;
        store = mr >= 0;
      }
      if (store && ep.row_zero != nullptr && ep.row_zero[orow]) zero = true;
      // per-column epilogue vectors of this tile -> smem while the main loop runs: every CTA reads the same few
      // cache lines at the same moment; from global inside the box loop that costs ~1 us of L2 queueing per box
      float* cv = colvec + acc * 1024;
      for (int c = threadIdx.x - 128; c < 256; c += 32 * EPI_WARPS) {
        const int gc = n_blk * BN + c;
        const bool ok = c < BN && gc < p.N;
        cv[c] = (ok && ep.col_bias != nullptr) ? __ldg(ep.col_bias + gc) : 0.f;
        cv[256 + c] = (ok && ep.col_scale != nullptr) ? __ldg(ep.col_scale + gc) : 1.f;
        cv[512 + c] = (ok && ep.slope1 != nullptr) ? __ldg(ep.slope1 + gc) : 1.f;
        cv[768 + c] = (ok && ep.slope2 != nullptr) ? __ldg(ep.slope2 + gc) : 1.f;
      }
      asm volatile("bar.sync 1, %0;" ::"n"(32 * EPI_WARPS) : "memory");

      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      if (warp == 4 && lane == 0) {
        if (it == 0) AVH_TRACE(6);
        AVH_TRACE(8);
      }
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * ACC_STRIDE;
      uint8_t* stg = epi_stage + (warp - 4) * 4096;

      if (p.c_mode != 0) {
        // ---- thread = row: TMEM -> registers -> fused math -> 128-byte-swizzled smem box -> TMA store / reduce-add
        const bool has_res = res_any && p.c_mode != 2;
        const int box_cols = out_f32 ? 32 : 64;
        const bool live = store && !zero;
        const int nboxes = (BN + box_cols - 1) / box_cols;
#pragma unroll 1
        for (int bx = half; bx < nboxes; bx += HSTRIDE) {
          const int cbase = bx * box_cols;                 // column offset inside the tile
          uint32_t packed[32];
#pragma unroll
          for (int sub = 0; sub < 2; ++sub) {
            if (sub == 1 && out_f32) break;
            const int c0 = cbase + sub * 32;
            const int col0 = n_blk * BN + c0;
            uint32_t rawv[32];
            if (c0 < BN) tmem_ld_32x32(taddr + c0, rawv);
            // residual row segment (32 columns) straight from global while the TMEM load is in flight
            uint4 rres[8];
            if (has_res && live && col0 < p.N) {
              if (out_f32) {
                const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(ep.R) + orow * ep.ldr + col0);
#pragma unroll
                for (int j = 0; j < 8; ++j) rres[j] = __ldg(rp + j);
              } else {
                const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(ep.R) + orow * ep.ldr + col0);
#pragma unroll
                for (int j = 0; j < 4; ++j) rres[j] = __ldg(rp + j);
              }
            }
            // stream-K owner: the first partial of this chunk is requested while the TMEM load is in flight (the
            // residual registers are free: stream-K is planned only for GEMMs without a separate residual operand)
            const bool sk_add = SK != 0 && c0 < BN && sk_last >= sk_first;
            if (sk_add) {
              const uint4* pp = reinterpret_cast<const uint4*>(p.sk_ws + ((size_t)sk_first * PAIR + cta_rank) * (size_t)BM * BN) +
                                (size_t)((c0 >> 5) * 8) * BM + q * 32 + lane;
#pragma unroll
              for (int j = 0; j < 8; ++j) rres[j] = __ldcg(pp + (size_t)j * BM);
            }
            tmem_ld_wait();
            float v[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = (c0 < BN) ? __uint_as_float(rawv[j]) : 0.f;
            if (sk_add) {
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                v[4 * j] += __uint_as_float(rres[j].x); v[4 * j + 1] += __uint_as_float(rres[j].y);
                v[4 * j + 2] += __uint_as_float(rres[j].z); v[4 * j + 3] += __uint_as_float(rres[j].w);
              }
              for (int pv = sk_first + 1; pv <= sk_last; ++pv) {       // further partials (K split over > 2 units), in order
                const float4* pp = reinterpret_cast<const float4*>(p.sk_ws + ((size_t)pv * PAIR + cta_rank) * (size_t)BM * BN) +
                                   (size_t)((c0 >> 5) * 8) * BM + q * 32 + lane;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  const float4 t4 = __ldcg(pp + (size_t)j * BM);
                  v[4 * j] += t4.x; v[4 * j + 1] += t4.y; v[4 * j + 2] += t4.z; v[4 * j + 3] += t4.w;
                }
              }
            }
            if (col0 < p.N) {
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float4 bi = *reinterpret_cast<const float4*>(cv + c0 + 4 * j);
                if (has_scale) {
                  const float4 sc = *reinterpret_cast<const float4*>(cv + 256 + c0 + 4 * j);
                  v[4 * j] = fmaf(v[4 * j], sc.x, bi.x); v[4 * j + 1] = fmaf(v[4 * j + 1], sc.y, bi.y);
                  v[4 * j + 2] = fmaf(v[4 * j + 2], sc.z, bi.z); v[4 * j + 3] = fmaf(v[4 * j + 3], sc.w, bi.w);
                } else {
                  v[4 * j] += bi.x; v[4 * j + 1] += bi.y; v[4 * j + 2] += bi.z; v[4 * j + 3] += bi.w;
                }
              }
              if (act == ACT_GELU) {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = gelu_erf_fast(v[j]);
              } else if (act == ACT_PRELU) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  const float4 s1 = *reinterpret_cast<const float4*>(cv + 512 + c0 + 4 * j);
                  v[4 * j] = v[4 * j] > 0.f ? v[4 * j] : v[4 * j] * s1.x;
                  v[4 * j + 1] = v[4 * j + 1] > 0.f ? v[4 * j + 1] : v[4 * j + 1] * s1.y;
                  v[4 * j + 2] = v[4 * j + 2] > 0.f ? v[4 * j + 2] : v[4 * j + 2] * s1.z;
                  v[4 * j + 3] = v[4 * j + 3] > 0.f ? v[4 * j + 3] : v[4 * j + 3] * s1.w;
                }
              }
              if (has_res && live) {
                if (out_f32) {
#pragma unroll
                  for (int j = 0; j < 8; ++j) {
                    v[4 * j] += __uint_as_float(rres[j].x); v[4 * j + 1] += __uint_as_float(rres[j].y);
                    v[4 * j + 2] += __uint_as_float(rres[j].z); v[4 * j + 3] += __uint_as_float(rres[j].w);
                  }
                } else {
#pragma unroll
                  for (int j = 0; j < 4; ++j) {
                    const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&rres[j]);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                      const float2 f = __bfloat1622float2(h2[k]);
                      v[8 * j + 2 * k] += f.x;
                      v[8 * j + 2 * k + 1] += f.y;
                    }
                  }
                }
              }
              if (has_s2) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  const float4 s2 = *reinterpret_cast<const float4*>(cv + 768 + c0 + 4 * j);
                  v[4 * j] = v[4 * j] > 0.f ? v[4 * j] : v[4 * j] * s2.x;
                  v[4 * j + 1] = v[4 * j + 1] > 0.f ? v[4 * j + 1] : v[4 * j + 1] * s2.y;
                  v[4 * j + 2] = v[4 * j + 2] > 0.f ? v[4 * j + 2] : v[4 * j + 2] * s2.z;
                  v[4 * j + 3] = v[4 * j + 3] > 0.f ? v[4 * j + 3] : v[4 * j + 3] * s2.w;
                }
              }
            }
            if (zero) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = 0.f;
            }
            if (out_f32) {
#pragma unroll
              for (int j = 0; j < 32; ++j) packed[j] = __float_as_uint(v[j]);
            } else {
#pragma unroll
              for (int j = 0; j < 16; ++j) packed[sub * 16 + j] = pack_bf16(v[2 * j], v[2 * j + 1]);
            }
          }
          if (bx + HSTRIDE >= nboxes) {
            // this warp's last TMEM read of the accumulator stage: hand it back to the MMA issuer
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              if (PAIR == 2) mbar_arrive_leader(&tmem_empty[acc]);
              else mbar_arrive(&tmem_empty[acc]);
            }
          }
          // the previous box of this warp must have been read out of smem before it is overwritten
          uint8_t* sbox = stg;
          if (lane == 0) tma_wait_group_read0();
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 8; ++j)
            *reinterpret_cast<uint4*>(sbox + lane * 128 + ((j ^ (lane & 7)) << 4)) =
                make_uint4(packed[4 * j], packed[4 * j + 1], packed[4 * j + 2], packed[4 * j + 3]);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            if (row0 < p.M) {
              if (p.c_mode == 2) tma_reduce_add_2d(&tma_c, sbox, n_blk * BN + cbase, row0);
              else tma_store_2d(&tma_c, sbox, n_blk * BN + cbase, row0);
            }
            tma_commit_group();       // one group per box, stored or not: "all but the newest group" = the box before
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
      } else {
        // ---- re-mapped rows: transpose 32x32 chunks through smem, then row-contiguous global accesses
        const uint32_t store_mask = __ballot_sync(0xffffffffu, store);
        const uint32_t zero_mask = __ballot_sync(0xffffffffu, zero);
        const int my_orow = (int)orow;
        float* stf = reinterpret_cast<float*>(stg);
        const int c4 = lane & 7, rsub = lane >> 3;
        const int nchunks = BN / 32;
#pragma unroll 1
        for (int ch = half; ch < nchunks; ch += HSTRIDE) {
          uint32_t rawv[32];
          tmem_ld_32x32(taddr + ch * 32, rawv);
          tmem_ld_wait();
          if (ch + HSTRIDE >= nchunks) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              if (PAIR == 2) mbar_arrive_leader(&tmem_empty[acc]);
              else mbar_arrive(&tmem_empty[acc]);
            }
          }
#pragma unroll
          for (int j = 0; j < 8; ++j)
            *reinterpret_cast<uint4*>(stf + lane * 32 + ((j ^ (lane & 7)) << 2)) =
                make_uint4(rawv[4 * j], rawv[4 * j + 1], rawv[4 * j + 2], rawv[4 * j + 3]);
          __syncwarp();
          const int col0 = n_blk * BN + ch * 32;
          if (col0 < p.N) {
            const int col = col0 + c4 * 4;
            const int cc = ch * 32 + c4 * 4;
            const float4 bi = *reinterpret_cast<const float4*>(cv + cc);
            const float4 sc = *reinterpret_cast<const float4*>(cv + 256 + cc);
            const float4 s1 = *reinterpret_cast<const float4*>(cv + 512 + cc);
            const float4 s2 = *reinterpret_cast<const float4*>(cv + 768 + cc);
#pragma unroll
            for (int g = 0; g < 2; ++g) {          // two groups of four rows: residual loads of a group in flight together
              long long orow4[4];
              float4 res[4];
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const int rr = (g * 4 + i) * 4 + rsub;
                orow4[i] = (long long)__shfl_sync(0xffffffffu, my_orow, rr);
                res[i] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (res_any && ((store_mask & ~zero_mask) >> rr) & 1u) {
                  const long long off = orow4[i] * ep.ldr + col;
                  if (out_f32) res[i] = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(ep.R) + off));
                  else {
                    const uint2 u = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(ep.R) + off));
                    const float2 f0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
                    const float2 f1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
                    res[i] = make_float4(f0.x, f0.y, f1.x, f1.y);
                  }
                }
              }
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const int rr = (g * 4 + i) * 4 + rsub;
                float4 v = *reinterpret_cast<const float4*>(stf + rr * 32 + ((c4 ^ (rr & 7)) << 2));
                if (has_scale) {
                  v.x = fmaf(v.x, sc.x, bi.x); v.y = fmaf(v.y, sc.y, bi.y);
                  v.z = fmaf(v.z, sc.z, bi.z); v.w = fmaf(v.w, sc.w, bi.w);
                } else {
                  v.x += bi.x; v.y += bi.y; v.z += bi.z; v.w += bi.w;
                }
                if (act == ACT_GELU) {
                  v.x = gelu_erf_fast(v.x); v.y = gelu_erf_fast(v.y); v.z = gelu_erf_fast(v.z); v.w = gelu_erf_fast(v.w);
                } else if (act == ACT_PRELU) {
                  v.x = v.x > 0.f ? v.x : v.x * s1.x; v.y = v.y > 0.f ? v.y : v.y * s1.y;
                  v.z = v.z > 0.f ? v.z : v.z * s1.z; v.w = v.w > 0.f ? v.w : v.w * s1.w;
                }
                if (res_any) { v.x += res[i].x; v.y += res[i].y; v.z += res[i].z; v.w += res[i].w; }
                if (has_s2) {
                  v.x = v.x > 0.f ? v.x : v.x * s2.x; v.y = v.y > 0.f ? v.y : v.y * s2.y;
                  v.z = v.z > 0.f ? v.z : v.z * s2.z; v.w = v.w > 0.f ? v.w : v.w * s2.w;
                }
                if ((zero_mask >> rr) & 1u) v = make_float4(0.f, 0.f, 0.f, 0.f);
                if ((store_mask >> rr) & 1u) {
                  const long long off = orow4[i] * ep.ldc + col;
                  if (out_f32) *reinterpret_cast<float4*>(reinterpret_cast<float*>(ep.C) + off) = v;
                  else *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(ep.C) + off) =
                           make_uint2(pack_bf16(v.x, v.y), pack_bf16(v.z, v.w));
                }
              }
            }
          }
          __syncwarp();      // staging buffer is rewritten by the next chunk
        }
        if (half >= nchunks) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (PAIR == 2) mbar_arrive_leader(&tmem_empty[acc]);
            else mbar_arrive(&tmem_empty[acc]);
          }
        }
      }
      if (warp == 4 && lane == 0) {
        if (it == 0) AVH_TRACE(7);
        AVH_TRACE(9);
      }
      if (SK != 0 && sk_last >= sk_first) {
        // every epilogue warp of this CTA has read its partial rows: hand the flags back (zero between launches)
        asm volatile("bar.sync 1, %0;" ::"n"(32 * EPI_WARPS) : "memory");
        if (threadIdx.x == 128)
          for (int v = sk_first; v <= sk_last; ++v) p.sk_flags[v * PAIR + cta_rank] = 0;
      }
    }
    if (lane == 0 && p.c_mode != 0) tma_wait_group0();     // bulk stores of this thread are complete
  }

  tc_fence_before();
  if (PAIR == 2) cluster_sync_all();
  else __syncthreads();
  tc_fence_after();
  if (threadIdx.x == 0) AVH_TRACE(10);
  if (warp == 2) {
    if (PAIR == 2) tmem_dealloc_pair(tmem_base, TMEM_COLS);
    else tmem_dealloc(tmem_base, TMEM_COLS);
    if (lane == 0) AVH_TRACE(11);
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

}  // namespace

// output tensor map: [rows, cols] fp32 or bf16, box = 128 bytes of columns x 32 rows, 128B swizzle
int encode_c(CUtensorMap* map, const void* base, long long rows, int cols, long long ld, int fp32) {
  EncodeTiledFn fn = get_encode_fn();
  AVH_CHECK(fn != nullptr, "cuTensorMapEncodeTiled entry point not available");
  const int es = fp32 ? 4 : 2;
  AVH_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0 && (ld * es) % 16 == 0, "TMA store alignment");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * es};
  cuuint32_t box[2] = {(cuuint32_t)(128 / es), 32u};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, fp32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                  const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  AVH_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (C) failed (code " + std::to_string((int)r) + ")");
  return 0;
}

// 2-D bf16 row-major tensor [rows, cols] (row stride ld elements), box = 64 cols x box_rows, 128B swizzle.
int encode_2d(CUtensorMap* map, const void* base, long long rows, int cols, long long ld, int box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  AVH_CHECK(fn != nullptr, "cuTensorMapEncodeTiled entry point not available");
  AVH_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0, "TMA base must be 16-byte aligned");
  AVH_CHECK((ld * 2) % 16 == 0, "TMA row stride must be a multiple of 16 bytes");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  AVH_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (code " + std::to_string((int)r) + ")");
  return 0;
}

namespace {

unsigned long long* g_trace = nullptr;

int default_pair() {
  static int v = -1;
  if (v < 0) {
    const char* e = std::getenv("AVH_GEMM_PAIR");
    v = (e != nullptr && e[0] == '2') ? 2 : 1;
  }
  return v;
}

// Modelled SM clocks of one launch (tools/gemm_stall.py, B200): a k-block of a 128 x bn tile needs 2 bn clk of tensor
// pipe, >= ~415 clk of issue + barrier handling, and (16 KB of A + 128 bn B of B) through the SM's L2 ingress at
// ~66 B/clk — the ingress bounds every single-CTA tile (bn 256: 785 clk measured, 192: 600-630, 160: 512-531); a CTA pair
// loads half of B per SM (bn 256: 537-544 clk, tensor-bound).  Around the main loop: ~3.2 kclk from entry to the first
// MMA (4.2 for pairs) and the exposed last epilogue (more for fp32 / reduce-add outputs, ~1.9x for pairs).  Persistent
// tiles run in whole rounds; stream-K (sk) gives every unit the same number of k-blocks + ~1.5 kclk of partial traffic.
double model_cycles(long long M, int N, int num_kb, int bn, int pair, int occ, int sms, int sk, int out_f32) {
  const long long mt = (M + (long long)BM * pair - 1) / ((long long)BM * pair);
  const long long nt = (N + bn - 1) / bn;
  const long long units = (long long)sms * occ / pair;
  const long long tiles = mt * nt;
  double kblock = 415.0;
  if (2.0 * bn > kblock) kblock = 2.0 * bn;
  const double ingress = occ * (double)(A_STAGE_BYTES + (bn / pair) * BK * 2) / 66.0;
  const double pipe = occ * 2.0 * bn;
  if (pipe > kblock) kblock = pipe;
  if (ingress > kblock) kblock = ingress;
  const double fill = pair == 2 ? 4200.0 : 3200.0;
  const double tail = (1500.0 + bn * (out_f32 ? 20.0 : 11.0)) * (pair == 2 ? 1.9 : 1.0);
  double main_loop;
  if (sk) {
    const long long U = tiles * num_kb;
    main_loop = (double)((U + units - 1) / units) * kblock + 1500.0;
  } else {
    main_loop = (double)((tiles + units - 1) / units) * (num_kb * kblock + 300.0);
  }
  return fill + main_loop + tail;
}

}  // namespace

void gemm_set_trace(unsigned long long* dev_buf) { g_trace = dev_buf; }

int gemm_plan(const GemmProblem& pr, GemmPlan* plan) {
  AVH_CHECK(pr.N % 32 == 0, "N must be a multiple of 32");
  AVH_CHECK(pr.num_kb >= 1, "num_kb must be >= 1");
  AVH_CHECK(pr.ktable == nullptr || pr.num_kb <= GEMM_MAX_KSTEPS, "too many K steps for the smem table");
  AVH_CHECK(pr.M >= 1 && pr.M < (1ll << 31) - 2 * BM, "M out of range");
  AVH_CHECK(pr.ep.C != nullptr, "output pointer is null");
  AVH_CHECK(pr.block_n >= 0 && pr.block_n <= 256 && pr.block_n % 32 == 0, "block_n must be a multiple of 32, <= 256");
  AVH_CHECK(pr.ep.R == nullptr || pr.ep.r_fp32 == pr.ep.c_fp32, "residual and output dtypes must match");
  plan->prob = pr;
  const int sms = device_sm_count();
  int pair = pr.pair ? pr.pair : default_pair();
  if (sms < 2) pair = 1;
  int bn = pr.block_n;
  int occ = pr.occ;
  if (pair == 2) occ = 1;
  // Stream-K is OFF unless AVH_GEMM_SK=1 (forced where applicable) or AVH_GEMM_SK=2 (cost model decides).  Measured at
  // M = 2400 (profiles/r2_gemm_streamk.txt): correct and bit-reproducible, but slower than whole tiles in rounds — qkv
  // 22.6 vs 18.1 us, fc1 22.0 vs 20.6, fc2 24.8 vs 23.0 (BN 160) — although it removes the idle part of the last round:
  // units at different k offsets no longer request the same A / B k-blocks at the same time, and the k-block time rises
  // by more than the balance gains.  Kept for shapes with very few tiles per SM (fc2 at BN 256: 29.7 vs 32.0 us).
  static int sk_env = -2;
  if (sk_env == -2) { const char* ev = std::getenv("AVH_GEMM_SK"); sk_env = ev ? std::atoi(ev) : 0; }
  if (sk_env == 2) sk_env = -1;      // -1 = model decides
  // stream-K needs the TMA epilogue (tile rows = output rows) and a workspace
  const Epilogue& e0 = pr.ep;
  const bool sk_possible = pr.sk_ws != nullptr && pr.sk_flags != nullptr && pr.streamk >= 0 && (sk_env != 0 || pr.streamk == 1) &&
                           e0.row_map == nullptr && e0.map_mode != MAP_2LEVEL && e0.row_zero == nullptr &&
                           (e0.R == nullptr || (e0.R == e0.C && e0.slope2 == nullptr && e0.c_fp32));
  int sk = 0;
  {
    double best = 1e30;
    int best_bn = bn, best_occ = occ ? occ : 1, best_sk = 0;
    const int step = pr.ep.c_fp32 ? 32 : 64;      // the TMA epilogue stores 128-byte boxes
    for (int oc = 1; oc <= 2; ++oc) {
      if (occ != 0 && oc != occ) continue;
      if (oc == 2 && pair == 2) continue;
      for (int c = step; c <= 256 / oc; c += step) {
        if (bn != 0 && c != bn) continue;
        if (bn == 0 && c > ((pr.N + step - 1) / step) * step) break;
        for (int k = 0; k <= 1; ++k) {
          if (k == 1) {
            if (!sk_possible || oc == 2 || (c % step) != 0 || pr.N % c != 0) continue;
            const long long units = (long long)sms / pair;
            const long long mt0 = (pr.M + (long long)BM * pair - 1) / ((long long)BM * pair);
            const long long tiles0 = mt0 * (pr.N / c);
            if (tiles0 % units == 0 || tiles0 * pr.num_kb < units) continue;          // nothing to balance
            if ((size_t)units * pair * BM * c * 4 > pr.sk_ws_bytes) continue;
          }
          if (k == 0 && (pr.streamk == 1 || sk_env == 1) && sk_possible) {
            // forced on: skip the persistent form when stream-K is applicable for this width
            const long long units = (long long)sms / pair;
            const long long mt0 = (pr.M + (long long)BM * pair - 1) / ((long long)BM * pair);
            if (oc == 1 && pr.N % c == 0 && (mt0 * (pr.N / c)) % units != 0 && mt0 * (pr.N / c) * pr.num_kb >= units &&
                (size_t)units * pair * BM * c * 4 <= pr.sk_ws_bytes)
              continue;
          }
          const double t = model_cycles(pr.M, pr.N, pr.num_kb, c, pair, oc, sms, k, pr.ep.c_fp32);
          if (t < best) { best = t; best_bn = c; best_occ = oc; best_sk = k; }
        }
      }
    }
    if (bn == 0) bn = best_bn;
    occ = (bn <= 128) ? best_occ : 1;
    sk = best_sk;
    if (bn == 0) { bn = 64; occ = 1; sk = 0; }
  }
  plan->prob.block_n = bn;
  plan->prob.pair = pair;
  plan->prob.occ = occ;
  plan->sk = sk;
  if (encode_2d(&plan->tma_a, pr.A, pr.a_rows, pr.a_cols, pr.lda, BM)) return 1;
  if (encode_2d(&plan->tma_b, pr.B, pr.b_rows, pr.b_cols, pr.ldb, bn / pair)) return 1;
  // TMA epilogue whenever tile rows map 1:1 onto output rows (Linear layers, implicit 3x3 convs, stem): plain
  // box stores, or reduce-add when the residual is the output itself (x += ...) and nothing follows the add
  {
    const Epilogue& e = pr.ep;
    const bool identity = e.row_map == nullptr &&
                          (e.map_mode != MAP_2LEVEL || (e.O2 == e.S2 && e.O1 == e.S1 && e.O0 == 0 && e.invalid_zero));
    int mode = 0;
    if (identity && (bn % (e.c_fp32 ? 32 : 64) == 0 || pr.N <= bn)) {
      mode = 1;
      if (e.R != nullptr && e.R == e.C) {
        // in-place residual: a reduce-add when nothing follows the add, else the per-thread path
        mode = (e.ldr == e.ldc && e.c_fp32 && e.slope2 == nullptr && e.row_zero == nullptr) ? 2 : 0;
      }
    }
    if (mode == 0) plan->sk = 0;
    plan->c_mode = mode;
    if (mode != 0) {
      if (encode_c(&plan->tma_c, e.C, pr.M, pr.N, e.ldc, e.c_fp32)) return 1;
    } else {
      plan->tma_c = plan->tma_a;
    }
  }
  const long long mt = (pr.M + (long long)BM * pair - 1) / ((long long)BM * pair);
  const long long nt = (pr.N + bn - 1) / bn;
  const long long tiles = mt * nt;
  const long long units = (long long)sms * occ / pair;
  plan->grid = (int)((tiles < units && !plan->sk) ? tiles : units) * pair;
  const int stage_bytes = A_STAGE_BYTES + (bn / pair) * BK * 2;
  const int ktab_bytes = pr.ktable != nullptr ? ((pr.num_kb * 16 + 1023) / 1024) * 1024 : 0;
  const int smem_limit = occ == 2 ? Occ<2>::SMEM_LIMIT : Occ<1>::SMEM_LIMIT;
  const int epi_bytes = occ == 2 ? Occ<2>::EPI_STAGE_BYTES : Occ<1>::EPI_STAGE_BYTES;
  int stages = (smem_limit - 1024 - epi_bytes - COLVEC_BYTES - ktab_bytes - BAR_BYTES) / stage_bytes;
  if (stages > MAX_STAGES) stages = MAX_STAGES;
  AVH_CHECK(stages >= 2, "tile too large for shared memory");
  plan->stages = stages;
  plan->ktab_bytes = ktab_bytes;
  plan->smem = 1024 + (size_t)stages * stage_bytes + epi_bytes + COLVEC_BYTES + ktab_bytes + BAR_BYTES;
  return 0;
}

int gemm_launch(const GemmPlan& plan, cudaStream_t stream) {
  const GemmProblem& pr = plan.prob;
  const int pair = pr.pair;
  KernelParams kp;
  kp.M = pr.M;
  kp.N = pr.N;
  kp.num_kb = pr.num_kb;
  kp.num_m_blk = (int)((pr.M + (long long)BM * pair - 1) / ((long long)BM * pair));
  kp.num_n_blk = (pr.N + pr.block_n - 1) / pr.block_n;
  kp.block_n = pr.block_n;
  kp.stages = plan.stages;
  kp.ktab_bytes = plan.ktab_bytes;
  kp.a_col_per_nblk = pr.a_col_per_nblk;
  kp.a_col_nblk = pr.a_col_nblk;
  kp.ktable = reinterpret_cast<const int4*>(pr.ktable);
  kp.c_mode = plan.c_mode;
  kp.sk = plan.sk;
  kp.sk_ws = pr.sk_ws;
  kp.sk_flags = pr.sk_flags;

  kp.trace = g_trace;
  kp.ep = pr.ep;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)plan.grid);
  const int occ = pr.occ == 2 ? 2 : 1;
  cfg.blockDim = dim3(occ == 2 ? Occ<2>::NUM_THREADS : Occ<1>::NUM_THREADS);
  cfg.dynamicSmemBytes = plan.smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)pair;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 2 : 1;
  const Epilogue& e = pr.ep;
  const int act = e.act, res = e.R != nullptr, s2 = e.slope2 != nullptr, scl = e.col_scale != nullptr, f32 = e.c_fp32;
  typedef void (*KernelFn)(CUtensorMap, CUtensorMap, CUtensorMap, KernelParams);
  KernelFn fn = nullptr;
  if (plan.sk != 0) {      // stream-K launches (AVH_GEMM_SK): single CTA per SM or CTA pairs, the three encoder epilogues
    if (pair == 2) fn = gemm_kernel<2, 1, -1, -1, -1, -1, -1, 1>;
    else if (act == ACT_NONE && !res && !s2 && !scl && !f32) fn = gemm_kernel<1, 1, ACT_NONE, 0, 0, 0, 0, 1>;
    else if (act == ACT_GELU && !res && !s2 && !scl && !f32) fn = gemm_kernel<1, 1, ACT_GELU, 0, 0, 0, 0, 1>;
    else if (act == ACT_NONE && res && !s2 && !scl && f32) fn = gemm_kernel<1, 1, ACT_NONE, 1, 0, 0, 1, 1>;
    else fn = gemm_kernel<1, 1, -1, -1, -1, -1, -1, 1>;
  }
#define AVH_SPEC(O, A, R, S, C, F)                                                                     \
  if (fn == nullptr && pair == 1 && occ == O && act == A && res == R && s2 == S && scl == C && f32 == F) \
    fn = gemm_kernel<1, O, A, R, S, C, F>;
  AVH_SPEC(1, ACT_NONE, 0, 0, 0, 0)      // Linear + bias -> bf16                  (qkv, modality projections)
  AVH_SPEC(1, ACT_NONE, 0, 0, 0, 1)      // Linear + bias -> fp32                  (post_extract_proj, fp32 mode)
  AVH_SPEC(1, ACT_GELU, 0, 0, 0, 0)      // Linear + bias + GELU -> bf16           (fc1)
  AVH_SPEC(1, ACT_GELU, 0, 0, 0, 1)      //                                        (fc1, fp32 mode)
  AVH_SPEC(1, ACT_NONE, 1, 0, 0, 1)      // Linear + bias + residual -> fp32       (out_proj, fc2)
  AVH_SPEC(1, ACT_GELU, 1, 0, 0, 1)      // conv + bias + GELU + residual -> fp32  (positional conv)
  AVH_SPEC(1, ACT_PRELU, 0, 0, 1, 0)     // conv + BN + PReLU -> bf16              (stem, block conv1)
  AVH_SPEC(1, ACT_PRELU, 0, 0, 1, 1)
  AVH_SPEC(1, ACT_NONE, 1, 1, 1, 0)      // conv + BN + residual + PReLU -> bf16   (block conv2)
  AVH_SPEC(1, ACT_NONE, 1, 1, 1, 1)
  AVH_SPEC(1, ACT_NONE, 0, 0, 1, 0)      // conv + BN -> bf16                      (downsample)
  AVH_SPEC(1, ACT_NONE, 0, 0, 1, 1)
  AVH_SPEC(2, ACT_NONE, 0, 0, 0, 0)      // two CTAs per SM: narrow tiles
  AVH_SPEC(2, ACT_NONE, 0, 0, 0, 1)
  AVH_SPEC(2, ACT_GELU, 0, 0, 0, 0)
  AVH_SPEC(2, ACT_NONE, 1, 0, 0, 1)
  AVH_SPEC(2, ACT_GELU, 1, 0, 0, 1)
  AVH_SPEC(2, ACT_PRELU, 0, 0, 1, 0)
  AVH_SPEC(2, ACT_NONE, 1, 1, 1, 0)
  AVH_SPEC(2, ACT_NONE, 0, 0, 1, 0)
#undef AVH_SPEC
  if (fn == nullptr) {
    if (pair == 2) fn = gemm_kernel<2, 1, -1, -1, -1, -1, -1>;
    else if (occ == 2) fn = gemm_kernel<1, 2, -1, -1, -1, -1, -1>;
    else fn = gemm_kernel<1, 1, -1, -1, -1, -1, -1>;
  }
  if (ensure_dyn_smem(reinterpret_cast<const void*>(fn), occ == 2 ? Occ<2>::SMEM_LIMIT : Occ<1>::SMEM_LIMIT)) return 1;
  AVH_CUDA_OK(cudaLaunchKernelEx(&cfg, fn, plan.tma_a, plan.tma_b, plan.tma_c, kp));
  count_launch(1);
  return 0;
}

}  // namespace avh
