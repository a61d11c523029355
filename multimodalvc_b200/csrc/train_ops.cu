// Training-mode pieces of the AV-HuBERT forward (SURVEY 8(a) row A18): what changes when the module is in .train() —
// as the frozen encoder of MMS-LLaMA is during training (src/model.py:280: no_grad, but never .eval()).
//
//  * BatchNorm with BATCH statistics (avhubert/resnet.py:23,44,56,139: nn.BatchNorm2d / 3d in training mode): the
//    convolution writes its raw output, bn_stats reduces per-channel sum and sum of squares (float64 partials,
//    one atomicAdd per CTA and channel), bn_finalize turns them into the normalising scale / bias (biased variance,
//    eps 1e-5) and updates running_mean / running_var (momentum, unbiased variance) exactly as torch does, bn_apply
//    normalises + PReLU (+ residual + PReLU) in place of the fused eval-mode epilogue.
//  * nn.Dropout (hubert.py:729 dropout_input; wav2vec2.py:879 after the positional conv; :980/:990 dropout1 / dropout3
//    on the block outputs before the residual add; :987 dropout2 = activation_dropout after the GELU): a
//    counter-based Philox4x32-10 stream keyed by (seed of the call, call-site id, element index) — every element's
//    mask is a pure function of those, so reruns with the same seed are bit-identical and no state is kept.
//    (The masks are NOT torch's: torch draws them from its own Philox offsets per kernel launch geometry.)
// LayerDrop (wav2vec2.py:887-888) is a host coin: the plan skips the layer's launches.
#include "common.cuh"
#include "kernels.h"
#include "philox.cuh"

#include <cuda_fp16.h>

namespace avh {
namespace {

__device__ __forceinline__ float ld_any(const void* p, int dt, long long i) {
  if (dt == DT_BF16) return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[i]);
  if (dt == DT_F16) return __half2float(reinterpret_cast<const __half*>(p)[i]);
  return reinterpret_cast<const float*>(p)[i];
}
__device__ __forceinline__ void st_any(void* out, int dt, long long i, float v) {
  if (dt == DT_BF16) reinterpret_cast<__nv_bfloat16*>(out)[i] = __float2bfloat16_rn(v);
  else if (dt == DT_F16) reinterpret_cast<__half*>(out)[i] = __float2half_rn(v);
  else reinterpret_cast<float*>(out)[i] = v;
}

// ---- per-channel sums over the rows of [rows, C]; rows with (r % period) >= valid are skipped (the gap frames of the
// stem's clip-padded row space; period = 0: no such gaps), and with S > 0 only the H x H image of the padded S x S layout.
// Thread = (row phase, group of 8 channels): one 16-byte (bf16) / two 16-byte (fp32) loads per row and thread, the row's
// validity worked out ONCE per row in 32-bit arithmetic (the first version did 64-bit divisions per element: 1.5 ms per
// BatchNorm at 8 clips), float64 partial sums per thread, one smem reduction and one double atomic per channel per CTA.
constexpr int BN_ROWS_PER_CTA = 2048;
// the per-channel double atomics of ~300 CTAs on 2 C addresses serialised (175 us per BatchNorm): CTAs spread their
// partial sums over BN_SLOTS copies of the accumulators, bn_finalize adds the copies
__global__ void __launch_bounds__(256)
bn_stats_kernel(const void* __restrict__ raw, int dt, long long rows, int C, long long period, long long valid, int S,
                int H, double* __restrict__ sums, int rows_per_cta) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ double sh[];                 // [phases][C][2]
  const int groups = C >> 3;                     // threads per row
  const int phases = 256 / groups > 0 ? 256 / groups : 1;
  const int gi = threadIdx.x % groups, ph = threadIdx.x / groups;
  const long long r0 = (long long)blockIdx.x * rows_per_cta;
  const long long r1 = r0 + rows_per_cta < rows ? r0 + rows_per_cta : rows;
  const unsigned int SS = (unsigned int)(S * S);
  for (int g0 = 0; g0 < groups; g0 += 256) {     // C > 2048 never happens; loop kept for generality
    const int g = g0 + gi;
    double a[8], q[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) { a[k] = 0.0; q[k] = 0.0; }
    if (ph < phases && g < groups) {
      // position of the row inside its period / image, advanced incrementally (no division in the loop but one 32-bit one)
      unsigned long long rp = period > 0 ? (unsigned long long)(r0 + ph) % (unsigned long long)period : 0ull;
      unsigned int rs = S > 0 ? (unsigned int)((unsigned long long)(r0 + ph) % SS) : 0u;
      for (long long r = r0 + ph; r < r1; r += phases) {
        const bool in_period = period <= 0 || rp < (unsigned long long)valid;
        bool in_image = true;
        if (S > 0) {
          const unsigned int y = rs / (unsigned int)S, x = rs - y * (unsigned int)S;
          in_image = y < (unsigned int)H && x < (unsigned int)H;
        }
        if (period > 0) { rp += phases; while (rp >= (unsigned long long)period) rp -= period; }
        if (S > 0) { rs += phases; while (rs >= SS) rs -= SS; }
        if (!in_period || !in_image) continue;
        float v[8];
        if (dt == DT_BF16) {
          const uint4 u = *reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(raw) + r * C + g * 8);
          const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
          for (int k = 0; k < 4; ++k) { const float2 f = __bfloat1622float2(h2[k]); v[2 * k] = f.x; v[2 * k + 1] = f.y; }
        } else if (dt == DT_F32) {
          const float4 u0 = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(raw) + r * C + g * 8);
          const float4 u1 = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(raw) + r * C + g * 8 + 4);
          v[0] = u0.x; v[1] = u0.y; v[2] = u0.z; v[3] = u0.w; v[4] = u1.x; v[5] = u1.y; v[6] = u1.z; v[7] = u1.w;
        } else {
#pragma unroll
          for (int k = 0; k < 8; ++k) v[k] = ld_any(raw, dt, r * C + g * 8 + k);
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) { a[k] += (double)v[k]; q[k] += (double)v[k] * (double)v[k]; }
      }
    }
    if (ph < phases && g < groups) {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        sh[((size_t)ph * C + g * 8 + k) * 2] = a[k];
        sh[((size_t)ph * C + g * 8 + k) * 2 + 1] = q[k];
      }
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += 256) {
      double ta = 0.0, tq = 0.0;
      for (int p2 = 0; p2 < phases; ++p2) { ta += sh[((size_t)p2 * C + c) * 2]; tq += sh[((size_t)p2 * C + c) * 2 + 1]; }
      double* slot = sums + (size_t)(blockIdx.x % BN_SLOTS) * 2 * C;
      atomicAdd(&slot[c], ta);
      atomicAdd(&slot[C + c], tq);
    }
    __syncthreads();
  }
}

// mean / biased variance -> scale, bias of the normalisation; running statistics updated like torch.nn.BatchNorm
__global__ void bn_finalize_kernel(double* __restrict__ sums, double count, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float eps, float momentum, float* __restrict__ rmean,
                                   float* __restrict__ rvar, float* __restrict__ scale, float* __restrict__ bias, int C) {
  pdl_launch_dependents();
  pdl_wait();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double s1 = 0.0, s2 = 0.0;
  for (int k = 0; k < BN_SLOTS; ++k) {
    double* slot = sums + (size_t)k * 2 * C;
    s1 += slot[c]; s2 += slot[C + c];
    slot[c] = 0.0; slot[C + c] = 0.0;      // ready for the next BatchNorm that uses this scratch
  }
  const double mean = s1 / count;
  double var = s2 / count - mean * mean;
  if (var < 0.0) var = 0.0;
  const float sc = gamma[c] * (float)(1.0 / sqrt(var + (double)eps));
  scale[c] = sc;
  bias[c] = beta[c] - (float)mean * sc;
  const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
  rmean[c] = (1.f - momentum) * rmean[c] + momentum * (float)mean;
  rvar[c] = (1.f - momentum) * rvar[c] + momentum * (float)unbiased;
}

// out = act2(act1(raw * scale + bias) + res); rows outside the H x H image of the padded S x S layout are zeros.
// Thread = 8 consecutive channels of one row (C % 8 == 0): 16-byte accesses, the row's validity computed once.
__global__ void __launch_bounds__(256)
bn_apply_kernel(const void* __restrict__ raw, void* __restrict__ out, int dt, long long rows, int C,
                const float* __restrict__ scale, const float* __restrict__ bias,
                const float* __restrict__ slope1, const void* __restrict__ res,
                const float* __restrict__ slope2, int S, int H) {
  pdl_launch_dependents();
  pdl_wait();
  const int groups = C >> 3;
  const long long gidx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gidx >= rows * groups) return;
  const long long r = gidx / groups;
  const int c0 = (int)(gidx - r * groups) * 8;
  bool ok = true;
  if (S > 0) {      // rows < 2^32 (checked by the launcher): 32-bit arithmetic
    const unsigned int rem = (unsigned int)r % (unsigned int)(S * S);
    const unsigned int y = rem / (unsigned int)S;
    ok = y < (unsigned int)H && rem - y * (unsigned int)S < (unsigned int)H;
  }
  const long long i0 = r * C + c0;
  float v[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) v[k] = 0.f;
  if (ok) {
    float x[8], rr[8];
    if (dt == DT_BF16) {
      const uint4 u = *reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(raw) + i0);
      const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
      for (int k = 0; k < 4; ++k) { const float2 f = __bfloat1622float2(h2[k]); x[2 * k] = f.x; x[2 * k + 1] = f.y; }
      if (res != nullptr) {
        const uint4 w = *reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(res) + i0);
        const __nv_bfloat162* g2 = reinterpret_cast<const __nv_bfloat162*>(&w);
#pragma unroll
        for (int k = 0; k < 4; ++k) { const float2 f = __bfloat1622float2(g2[k]); rr[2 * k] = f.x; rr[2 * k + 1] = f.y; }
      }
    } else {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        x[k] = ld_any(raw, dt, i0 + k);
        rr[k] = res != nullptr ? ld_any(res, dt, i0 + k) : 0.f;
      }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float t = fmaf(x[k], scale[c0 + k], bias[c0 + k]);
      if (slope1 != nullptr) t = t > 0.f ? t : t * slope1[c0 + k];
      if (res != nullptr) t += rr[k];
      if (slope2 != nullptr) t = t > 0.f ? t : t * slope2[c0 + k];
      v[k] = t;
    }
  }
  if (dt == DT_BF16) {
    uint4 u;
    __nv_bfloat162* h2 = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
    for (int k = 0; k < 4; ++k) h2[k] = __floats2bfloat162_rn(v[2 * k], v[2 * k + 1]);
    *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(out) + i0) = u;
  } else {
#pragma unroll
    for (int k = 0; k < 8; ++k) st_any(out, dt, i0 + k, v[k]);
  }
}

// x = dropout(x) in place, or x += dropout(t) when `add` is given (dropout1 / dropout3 before the residual add)
__global__ void dropout_kernel(void* __restrict__ x, int dt, const float* __restrict__ add, long long n, float p,
                               unsigned long long seed, unsigned int site) {
  pdl_launch_dependents();
  pdl_wait();
  const long long i4 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long base = i4 * 4;
  if (base >= n) return;
  const uint4 rnd = philox4x32(seed, (unsigned long long)i4, site);
  const unsigned int rv[4] = {rnd.x, rnd.y, rnd.z, rnd.w};
  const float keep = 1.f / (1.f - p);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const long long i = base + k;
    if (i >= n) break;
    const float m = u01(rv[k]) >= p ? keep : 0.f;
    if (add != nullptr) {
      float* xf = reinterpret_cast<float*>(x);
      xf[i] += add[i] * m;
    } else {
      st_any(x, dt, i, ld_any(x, dt, i) * m);
    }
  }
}

inline int blocks_for(long long n, int per) { return (int)((n + per - 1) / per); }

}  // namespace

int launch_bn_stats(const void* raw, int dt, long long rows, int C, long long period, long long valid, int S, int H,
                    double* sums, cudaStream_t stream) {
  AVH_CHECK(C >= 8 && C % 8 == 0 && C <= 2048 && (C / 8 <= 256 ? 256 % (C / 8) == 0 : false),
            "bn_stats: channel count must be a multiple of 8 whose 8-channel groups divide 256");
  if (rows <= 0) return 0;
  const int phases = 256 / (C / 8);
  const size_t smem = (size_t)phases * C * 2 * sizeof(double);
  AVH_CHECK(smem <= 48 * 1024, "bn_stats: shared-memory reduction buffer too large");
  // rows per CTA: enough CTAs to fill the machine (a thread has ONE 16-byte load in flight: the small maps of layers 3-4
  // gave 10-30 CTAs at 2048 rows each and ran at a few GB/s per CTA), never more than BN_ROWS_PER_CTA
  long long rpc = (rows + 4 * 148 - 1) / (4 * 148);
  rpc = (rpc + phases - 1) / phases * phases;
  if (rpc < 4 * phases) rpc = 4 * phases;
  if (rpc > BN_ROWS_PER_CTA) rpc = BN_ROWS_PER_CTA;
  AVH_CUDA_OK(launch_pdl(bn_stats_kernel, dim3(blocks_for(rows, (int)rpc)), dim3(256), smem, stream, raw, dt, rows, C,
                         period, valid, S, H, sums, (int)rpc));
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_bn_finalize(double* sums, double count, const float* gamma, const float* beta, float eps, float momentum,
                       float* rmean, float* rvar, float* scale, float* bias, int C, cudaStream_t stream) {
  AVH_CUDA_OK(launch_pdl(bn_finalize_kernel, dim3(blocks_for(C, 128)), dim3(128), 0, stream, sums, count, gamma, beta, eps,
                         momentum, rmean, rvar, scale, bias, C));
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_bn_apply(const void* raw, void* out, int dt, long long rows, int C, const float* scale, const float* bias,
                    const float* slope1, const void* res, const float* slope2, int S, int H, cudaStream_t stream) {
  const long long n = rows * C;
  if (n <= 0) return 0;
  AVH_CHECK(C % 8 == 0 && rows < (1ll << 32), "bn_apply: channel count must be a multiple of 8, rows < 2^32");
  AVH_CUDA_OK(launch_pdl(bn_apply_kernel, dim3(blocks_for(n / 8, 256)), dim3(256), 0, stream, raw, out, dt, rows, C, scale, bias,
                         slope1, res, slope2, S, H));
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_dropout(void* x, int dt, const float* add, long long n, float p, unsigned long long seed, unsigned int site,
                   cudaStream_t stream) {
  AVH_CHECK(p >= 0.f && p < 1.f, "dropout probability must be in [0, 1)");
  AVH_CHECK(add == nullptr || dt == DT_F32, "dropout_add accumulates into an fp32 tensor");
  if (n <= 0) return 0;
  AVH_CUDA_OK(launch_pdl(dropout_kernel, dim3(blocks_for((n + 3) / 4, 256)), dim3(256), 0, stream, x, dt, add, n, p, seed, site));
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

}  // namespace avh
