// 3x3 / stride-1 / 64 -> 64 channel convolution (+ folded BatchNorm, PReLU, residual, PReLU) on tcgen05 with the
// operand WINDOW resident in shared memory: the layer1 convolutions of the lip ResNet (avhubert/resnet.py:35-74 with
// planes = 64; 22 % of the frontend's FLOPs and, as a 9-tap shifted-row GEMM with N = 64, bound by the L2->SM operand
// stream: every tap re-fetched its own 128-row A tile and the 8 KB weight slice).
//
// Layout: activations NHWC with one shared zero row/column per image, flat [n*S*S, 64] (S = H + 1).  For a tile of
// 128 consecutive rows [m0, m0+128) the nine taps read rows m0 + (kh-1)*S + (kw-1) + i, i.e. nine overlapping
// 128-row slices of ONE window [m0 - S - 1, m0 + 128 + S + 1).  The window is loaded once by TMA (128-byte swizzle,
// out-of-bounds rows zero-filled); each tap's A operand is a UMMA descriptor whose start address is the window base
// plus (kh*S + kw) * 128 B — legal because the 128-byte swizzle is a function of the absolute smem address
// (tools/micro/desc_offset.cu).  The 9 x 64 x 64 weights (72 KB) are loaded once per CTA and stay resident.
// Per tile: 1 TMA load (22.5 KB for S = 23) and 36 tcgen05.mma of 128 x 64 x 16.
//
// Roles as in gemm_tcgen05.cu: warp 0 TMA producer, warp 1 MMA issuer (elected lane, warp-uniform loop), warp 2 TMEM
// allocator, warps 4-11 epilogue in two sets that alternate tiles (thread = row: tcgen05.ld -> scale/bias/PReLU/residual/PReLU, zero pad rows ->
// swizzled smem box -> TMA store).
#include "common.cuh"
#include "gemm.h"

#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <set>
#include <vector>

namespace avh {
namespace {

constexpr int BM = 128;
constexpr int CH = 64;                         // channels in = channels out
constexpr int B_TAP_BYTES = CH * CH * 2;       // 8 KB per tap
constexpr int B_BYTES = 9 * B_TAP_BYTES;       // 72 KB resident weights
constexpr int NUM_THREADS = 384;               // producer, mma, alloc, spare + 2 sets of 4 epilogue warps
constexpr int EPI_BYTES = 8 * 4096;
constexpr int MAX_STAGES = 6;
constexpr int SMEM_LIMIT = 227 * 1024;

struct WinParams {
  long long rows;
  int S;
  int num_tiles;
  int stages;
  int win_rows;          // 128 + 2 * (S + 1)
  int win_bytes;         // win_rows * 128 rounded up to 1024
  const float* scale;
  const float* bias;
  const float* slope1;
  const float* slope2;
  const __nv_bfloat16* R;
  unsigned long long* dbg;     // debug (AVH_WIN_DBG=1): per CTA 8 stall counters in SM clocks, else null
};

__device__ __forceinline__ void wait_dbg(uint64_t* bar, uint32_t parity, unsigned long long* dbg, long long& acc) {
  if (dbg == nullptr) { mbar_wait(bar, parity); return; }
  const long long c0 = clock64();
  mbar_wait(bar, parity);
  acc += clock64() - c0;
}

// The stall counters (AVH_WIN_DBG=1) show the producer waiting for free stages 78 % of the time and the MMA warp busy
// 93 %: ~64 clk per 128 x 64 x 16 MMA, i.e. the tensor core is fed at half rate — an SS-form MMA with N = 64 re-reads
// its 4 KB A slice from shared memory for only 64 output columns (the same bound the first fused stem hit).  Running
// each tap as one 256-row MMA of a CTA pair does not lift that bound (DESIGN.md, tried and rejected).
template <bool RES>
__global__ void __launch_bounds__(NUM_THREADS, 1)
conv_window_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                   const __grid_constant__ CUtensorMap tma_c, const WinParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  uint8_t* smem_b = smem;
  uint8_t* smem_a = smem + B_BYTES;
  uint8_t* epi_stage = smem_a + p.stages * p.win_bytes;
  float* colvec = reinterpret_cast<float*>(epi_stage + EPI_BYTES);     // scale | bias | slope1 | slope2, 64 each
  uint64_t* b_full = reinterpret_cast<uint64_t*>(colvec + 4 * CH);
  uint64_t* a_full = b_full + 1;
  uint64_t* a_empty = a_full + MAX_STAGES;
  uint64_t* tmem_full = a_empty + MAX_STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int unit = blockIdx.x, num_units = gridDim.x;      // persistent CTAs: tiles unit, unit + num_units, ...
  pdl_launch_dependents();
  const long long k_start = clock64();
  long long st0 = 0, st1 = 0;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
    tma_prefetch_desc(&tma_c);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(b_full, 1);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&a_full[s], 1);
      mbar_init(&a_empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], 4);
    }
    mbar_fence_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, 128);
  if (threadIdx.x < CH) {           // launch-constant per-channel vectors
    const int c = threadIdx.x;
    colvec[c] = __ldg(p.scale + c);
    colvec[CH + c] = __ldg(p.bias + c);
    colvec[2 * CH + c] = p.slope1 != nullptr ? __ldg(p.slope1 + c) : 1.f;
    colvec[3 * CH + c] = p.slope2 != nullptr ? __ldg(p.slope2 + c) : 1.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (warp == 0) {                  // the resident weights are launch constants: request them before the wait
    if (elect_one()) {
      mbar_expect_tx(b_full, B_BYTES);
      for (int t = 0; t < 9; ++t) tma_load_2d(smem_b + t * B_TAP_BYTES, &tma_b, b_full, t * CH, 0);
    }
    __syncwarp();
  }
  pdl_wait();                       // from here on: activations of the previous kernel

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = unit; tile < p.num_tiles; tile += num_units) {
      wait_dbg(&a_empty[stage], phase ^ 1, p.dbg, st0);
      if (elect_one()) {
        mbar_expect_tx(&a_full[stage], (uint32_t)p.win_rows * 128u);
        tma_load_2d(smem_a + stage * p.win_bytes, &tma_a, &a_full[stage], 0, tile * BM - p.S - 1);
      }
      __syncwarp();
      if (++stage == p.stages) { stage = 0; phase ^= 1; }
    }
    if (p.dbg != nullptr && lane == 0) p.dbg[blockIdx.x * 8 + 1] = st0;
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc = umma_idesc_bf16(BM, CH);
    mbar_wait(b_full, 0);
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int tile = unit; tile < p.num_tiles; tile += num_units, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      wait_dbg(&tmem_empty[acc], acc_phase ^ 1, p.dbg, st0);
      wait_dbg(&a_full[stage], phase, p.dbg, st1);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + acc * CH;
      const uint32_t a_base = smem_u32(smem_a + stage * p.win_bytes);
      const uint32_t b_base = smem_u32(smem_b);
      if (elect_one()) {
#pragma unroll
        for (int t = 0; t < 9; ++t) {
          // tap (kh, kw): rows of the window starting at kh*S + kw
          const uint64_t adesc = umma_desc_sw128(a_base + (uint32_t)((t / 3) * p.S + (t % 3)) * 128u);
          const uint64_t bdesc = umma_desc_sw128(b_base + t * B_TAP_BYTES);
#pragma unroll
          for (int k = 0; k < CH / 16; ++k) umma_bf16(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (t | k) != 0);
        }
        umma_commit(&a_empty[stage]);
        umma_commit(&tmem_full[acc]);
      }
      __syncwarp();
      if (++stage == p.stages) { stage = 0; phase ^= 1; }
    }
    if (p.dbg != nullptr && lane == 0) { p.dbg[blockIdx.x * 8 + 2] = st0; p.dbg[blockIdx.x * 8 + 3] = st1; p.dbg[blockIdx.x * 8 + 6] = it; }
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ epilogue: thread = row
    // two warp sets alternate tiles (set e owns accumulator stage e), so each set has two tile times for its epilogue
    const int q = warp & 3;
    const int eset = (warp - 4) >> 2;
    uint8_t* stg = epi_stage + (warp - 4) * 4096;
    const int S = p.S, H = p.S - 1;
    int it = 0;
    for (int tile = unit; tile < p.num_tiles; tile += num_units, ++it) {
      if ((it & 1) != eset) continue;
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int row0 = tile * BM + q * 32;
      const long long r = (long long)row0 + lane;
      const bool inside = r < p.rows;
      const int rem = (int)(r % (S * S));
      const int hh = rem / S, ww = rem - hh * S;
      const bool valid = inside && hh < H && ww < H;      // pad rows/columns of the layout are written as zeros
      uint4 rres[8];
      if (RES && valid) {                                 // residual row (128 B) in flight before the accumulator is ready
        const uint4* rp = reinterpret_cast<const uint4*>(p.R + r * CH);
#pragma unroll
        for (int j = 0; j < 8; ++j) rres[j] = __ldg(rp + j);
      }
      wait_dbg(&tmem_full[acc], acc_phase, p.dbg, st0);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * CH;
      uint32_t packed[32];
#pragma unroll
      for (int sub = 0; sub < 2; ++sub) {
        uint32_t rawv[32];
        tmem_ld_32x32(taddr + sub * 32, rawv);
        tmem_ld_wait();
        if (sub == 1) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tmem_empty[acc]);
        }
        float v[32];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 sc = *reinterpret_cast<const float4*>(colvec + sub * 32 + 4 * j);
          const float4 bi = *reinterpret_cast<const float4*>(colvec + CH + sub * 32 + 4 * j);
          v[4 * j] = fmaf(__uint_as_float(rawv[4 * j]), sc.x, bi.x);
          v[4 * j + 1] = fmaf(__uint_as_float(rawv[4 * j + 1]), sc.y, bi.y);
          v[4 * j + 2] = fmaf(__uint_as_float(rawv[4 * j + 2]), sc.z, bi.z);
          v[4 * j + 3] = fmaf(__uint_as_float(rawv[4 * j + 3]), sc.w, bi.w);
        }
        if (!RES) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 s1 = *reinterpret_cast<const float4*>(colvec + 2 * CH + sub * 32 + 4 * j);
            v[4 * j] = v[4 * j] > 0.f ? v[4 * j] : v[4 * j] * s1.x;
            v[4 * j + 1] = v[4 * j + 1] > 0.f ? v[4 * j + 1] : v[4 * j + 1] * s1.y;
            v[4 * j + 2] = v[4 * j + 2] > 0.f ? v[4 * j + 2] : v[4 * j + 2] * s1.z;
            v[4 * j + 3] = v[4 * j + 3] > 0.f ? v[4 * j + 3] : v[4 * j + 3] * s1.w;
          }
        } else {
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
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 s2 = *reinterpret_cast<const float4*>(colvec + 3 * CH + sub * 32 + 4 * j);
            v[4 * j] = v[4 * j] > 0.f ? v[4 * j] : v[4 * j] * s2.x;
            v[4 * j + 1] = v[4 * j + 1] > 0.f ? v[4 * j + 1] : v[4 * j + 1] * s2.y;
            v[4 * j + 2] = v[4 * j + 2] > 0.f ? v[4 * j + 2] : v[4 * j + 2] * s2.z;
            v[4 * j + 3] = v[4 * j + 3] > 0.f ? v[4 * j + 3] : v[4 * j + 3] * s2.w;
          }
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) packed[sub * 16 + j] = valid ? pack_bf16(v[2 * j], v[2 * j + 1]) : 0u;
      }
      if (lane == 0) tma_wait_group_read0();      // previous box of this warp has left smem
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 8; ++j)
        *reinterpret_cast<uint4*>(stg + lane * 128 + ((j ^ (lane & 7)) << 4)) =
            make_uint4(packed[4 * j], packed[4 * j + 1], packed[4 * j + 2], packed[4 * j + 3]);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0 && row0 < p.rows) {
        tma_store_2d(&tma_c, stg, 0, row0);       // rows beyond the tensor are clipped by TMA
        tma_commit_group();
      }
    }
    if (lane == 0) tma_wait_group0();
    if (p.dbg != nullptr && lane == 0 && (warp == 4 || warp == 8)) p.dbg[blockIdx.x * 8 + 4 + ((warp - 4) >> 2)] = st0;
  }

  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 2) tmem_dealloc(tmem_base, 128);
  if (p.dbg != nullptr && threadIdx.x == 0) p.dbg[blockIdx.x * 8] = clock64() - k_start;
}

}  // namespace

int conv_window_plan(const ConvWinProblem& pr, ConvWinPlan* plan) {
  AVH_CHECK(pr.A && pr.B && pr.C && pr.scale && pr.bias, "null pointer");
  AVH_CHECK(pr.S >= 2 && pr.S <= 60, "unsupported image pitch");
  AVH_CHECK(pr.rows >= 1 && pr.rows < (1ll << 31) - 1024, "rows out of range");
  plan->prob = pr;
  plan->win_rows = BM + 2 * (pr.S + 1);
  AVH_CHECK(plan->win_rows <= 256, "window exceeds the TMA box limit");
  const int win_bytes = ((plan->win_rows * 128 + 1023) / 1024) * 1024;
  const int fixed = 1024 + B_BYTES + EPI_BYTES + 4 * CH * 4 + (1 + 2 * MAX_STAGES + 4) * 8 + 16;
  int stages = (SMEM_LIMIT - fixed) / win_bytes;
  if (stages > MAX_STAGES) stages = MAX_STAGES;
  AVH_CHECK(stages >= 2, "window too large for shared memory");
  plan->stages = stages;
  plan->smem = (size_t)fixed + (size_t)stages * win_bytes;
  if (encode_2d(&plan->tma_a, pr.A, pr.rows, CH, CH, plan->win_rows)) return 1;
  if (encode_2d(&plan->tma_b, pr.B, CH, 9 * CH, 9 * CH, CH)) return 1;
  if (encode_c(&plan->tma_c, pr.C, pr.rows, CH, CH, 0)) return 1;
  const long long tiles = (pr.rows + BM - 1) / BM;
  const long long sms = device_sm_count();
  plan->grid = (int)(tiles < sms ? tiles : sms);
  return 0;
}

int conv_window_launch(const ConvWinPlan& plan, cudaStream_t stream) {
  const ConvWinProblem& pr = plan.prob;
  WinParams p;
  p.rows = pr.rows;
  p.S = pr.S;
  p.num_tiles = (int)((pr.rows + BM - 1) / BM);
  p.stages = plan.stages;
  p.win_rows = plan.win_rows;
  p.win_bytes = ((plan.win_rows * 128 + 1023) / 1024) * 1024;
  p.scale = pr.scale;
  p.bias = pr.bias;
  p.slope1 = pr.slope1;
  p.slope2 = pr.slope2;
  p.R = reinterpret_cast<const __nv_bfloat16*>(pr.R);
  typedef void (*WinFn)(CUtensorMap, CUtensorMap, CUtensorMap, WinParams);
  WinFn fn = pr.R != nullptr ? conv_window_kernel<true> : conv_window_kernel<false>;
  if (ensure_dyn_smem(reinterpret_cast<const void*>(fn), SMEM_LIMIT)) return 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)plan.grid);
  cfg.blockDim = dim3(NUM_THREADS);
  cfg.dynamicSmemBytes = plan.smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 2 : 1;
  p.dbg = nullptr;
  static int dbg_env = -1;
  if (dbg_env < 0) { const char* ev = std::getenv("AVH_WIN_DBG"); dbg_env = ev != nullptr ? std::atoi(ev) : 0; }
  if (dbg_env > 0) {
    // debug only: stall accounting of one launch (synchronises the stream), printed to stderr
    --dbg_env;
    unsigned long long* d = nullptr;
    AVH_CUDA_OK(cudaMalloc(&d, (size_t)plan.grid * 64));
    AVH_CUDA_OK(cudaMemset(d, 0, (size_t)plan.grid * 64));
    p.dbg = d;
    AVH_CUDA_OK(cudaLaunchKernelEx(&cfg, fn, plan.tma_a, plan.tma_b, plan.tma_c, p));
    AVH_CUDA_OK(cudaStreamSynchronize(stream));
    std::vector<unsigned long long> hst((size_t)plan.grid * 8);
    AVH_CUDA_OK(cudaMemcpy(hst.data(), d, (size_t)plan.grid * 64, cudaMemcpyDeviceToHost));
    cudaFree(d);
    static const char* names[8] = {"total", "prod_wait_empty", "mma_wait_tmem_empty", "mma_wait_a_full", "epi0_wait_full",
                                   "epi1_wait_full", "tiles", "-"};
    for (int c : {0, plan.grid / 2, plan.grid - 1}) {
      std::fprintf(stderr, "[conv_window dbg] res=%d cta %d:", pr.R != nullptr, c);
      for (int i = 0; i < 7; ++i) std::fprintf(stderr, " %s=%llu", names[i], hst[(size_t)c * 8 + i]);
      std::fprintf(stderr, "\n");
    }
    count_launch(1);
    return 0;
  }
  AVH_CUDA_OK(cudaLaunchKernelEx(&cfg, fn, plan.tma_a, plan.tma_b, plan.tma_c, p));
  count_launch(1);
  return 0;
}

}  // namespace avh
