// Backward of the Transformer encoder (SURVEY 8(a) row A18 / BASELINE config 5, encoder part): everything that is not a
// GEMM.  The four contractions of every Linear's backward run on the tcgen05 GEMM of gemm_tcgen05.cu:
//   dX = dY W        -> A = dY [tokens, out] (operand form), B = W^T packed K-major at weight-finalisation time
//   dW = dY^T X      -> A = dY^T [out, tokens], B = X^T [in, tokens]: both produced by transpose_split (K = tokens, zero
//                       padded to a multiple of 64; in the fp32-faithful mode as bf16 hi + mid planes like every operand)
//   db = column sums of dY
// and the kernels below are the element-wise / row-wise / attention parts, fp32 arithmetic, deterministic (no atomics):
//   gelu_fwd / gelu_bwd        erf GELU and its derivative Phi(u) + u phi(u)      (fairseq/fairseq/modules/gelu.py:95-96)
//   ln_stats + ln_bwd_dx + ln_bwd_params   LayerNorm backward (fairseq/fairseq/modules/layer_norm.py:51-56 -> F.layer_norm)
//   ln_post_bwd_dx             the post-LN form: LN^T(residual-path + block-path gradient), with the masked gradient of
//                               the block that feeds the LayerNorm and its GEMM operand planes in the same pass
//   attention_bwd_dq / attention_bwd_dkv  softmax attention backward with the probabilities recomputed from the saved
//                               log-sum-exp of every query row (fairseq/fairseq/modules/multihead_attention.py:170-192)
#include "attn_tile.cuh"
#include "common.cuh"
#include "kernels.h"
#include "philox.cuh"

#include <cuda_fp16.h>

namespace avh {
namespace {

__device__ __forceinline__ float ldb(const void* p, int dt, long long i) {
  if (dt == DT_BF16) return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[i]);
  if (dt == DT_F16) return __half2float(reinterpret_cast<const __half*>(p)[i]);
  return reinterpret_cast<const float*>(p)[i];
}
__device__ __forceinline__ void stb(void* out, int dt, long long i, float v) {
  if (dt == DT_BF16) reinterpret_cast<__nv_bfloat16*>(out)[i] = __float2bfloat16_rn(v);
  else if (dt == DT_F16) reinterpret_cast<__half*>(out)[i] = __float2half_rn(v);
  else reinterpret_cast<float*>(out)[i] = v;
}

// in [rows, C] (row stride ld, any float dtype) -> out bf16 [C, planes * kpad]: out[c, p * kpad + r] = plane p of in[r, c]
// (plane 0 = bf16 round, plane 1 = bf16 of the remainder); columns r in [rows, kpad) are zero.  32 x 32 tiles through smem.
__global__ void __launch_bounds__(256)
transpose_split_kernel(const void* __restrict__ in, int dt, long long ld, long long rows, int C, __nv_bfloat16* __restrict__ out,
                       int planes, long long kpad, float scale, int T, int Tp, long long out_ld) {
  __shared__ float tile[32][33];
  const long long r0 = (long long)blockIdx.x * 32;      // OUTPUT column (= K index) of the tile
  const int c0 = blockIdx.y * 32;
  for (int k = threadIdx.x; k < 1024; k += 256) {
    const int i = k / 32, j = k % 32;            // i = row in tile, j = column in tile (coalesced along columns)
    long long r = r0 + i;
    const int c = c0 + j;
    bool live = true;
    if (T > 0) {                                 // zero-gapped time layout: K index (b * Tp + t) <- input row b * T + t
      const long long bb = r / Tp;
      const int t = (int)(r % Tp);
      live = t < T;
      r = bb * T + t;
    }
    tile[i][j] = (live && r < rows && c < C) ? ldb(in, dt, r * ld + c) * scale : 0.f;
  }
  __syncthreads();
  for (int k = threadIdx.x; k < 1024; k += 256) {
    const int j = k / 32, i = k % 32;            // output row = column c0 + j, output column = r0 + i (coalesced)
    const int c = c0 + j;
    const long long r = r0 + i;
    if (c >= C || r >= kpad) continue;
    const float v = tile[i][j];
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    out[(long long)c * out_ld + r] = hi;
    if (planes > 1) out[(long long)c * out_ld + kpad + r] = __float2bfloat16_rn(v - __bfloat162float(hi));
  }
}

// out[c] = scale * sum_r in[r, c]: one CTA per 32 columns, 8 row phases, fixed summation order
constexpr int CS_PH = 32;      // row phases of the column reductions (1024 threads = 32 columns x 32 phases)
__global__ void __launch_bounds__(1024)
colsum_kernel(const void* __restrict__ in, int dt, long long ld, long long rows, int C, float* __restrict__ out, float scale) {
  __shared__ float part[CS_PH][33];
  const int j = threadIdx.x % 32, ph = threadIdx.x / 32;
  const int c = blockIdx.x * 32 + j;
  float s = 0.f;
  if (c < C)
    for (long long r = ph; r < rows; r += CS_PH) s += ldb(in, dt, r * ld + c);
  part[ph][j] = s;
  __syncthreads();
  if (ph == 0 && c < C) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < CS_PH; ++k) t += part[k][j];
    out[c] = t * scale;
  }
}

__device__ __forceinline__ float gelu_erf(float u) { return 0.5f * u * (1.f + erff(u * 0.70710678118654752f)); }
__device__ __forceinline__ float gelu_grad(float u) {
  const float cdf = 0.5f * (1.f + erff(u * 0.70710678118654752f));
  const float pdf = 0.3989422804014327f * __expf(-0.5f * u * u);
  return cdf + u * pdf;
}

// out = (res ? res : 0) + gelu(u)
__global__ void __launch_bounds__(256)
gelu_fwd_kernel(const void* __restrict__ u, int u_dt, const float* __restrict__ res, void* __restrict__ out, int out_dt, long long n) {
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const float v = gelu_erf(ldb(u, u_dt, i)) + (res ? res[i] : 0.f);
    stb(out, out_dt, i, v);
  }
}
// du = dg * gelu'(u)
__global__ void __launch_bounds__(256)
gelu_bwd_kernel(const void* __restrict__ u, int u_dt, const void* __restrict__ dg, int dg_dt, void* __restrict__ du, int du_dt, long long n) {
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256)
    stb(du, du_dt, i, ldb(dg, dg_dt, i) * gelu_grad(ldb(u, u_dt, i)));
}

__device__ __forceinline__ float wsum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// LayerNorm backward w.r.t. the input, warp per row: xhat = (x - mean) rstd, g = dy gamma,
// dx = rstd (g - mean(g) - xhat mean(g xhat)); out = (res ? res : 0) + dx.  Also stores (mean, rstd) per row for the
// parameter-gradient kernel.
__global__ void __launch_bounds__(256)
ln_bwd_dx_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ dy,
                 const float* __restrict__ res, float* __restrict__ out, float2* __restrict__ stats, long long rows, int C,
                 float eps) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + row * C;
  const float* dr = dy + row * C;
  float s = 0.f;
  for (int c = lane; c < C; c += 32) s += xr[c];
  const float mean = wsum(s) / C;
  float q = 0.f;
  for (int c = lane; c < C; c += 32) { const float d = xr[c] - mean; q += d * d; }
  const float rstd = rsqrtf(wsum(q) / C + eps);
  float a = 0.f, b = 0.f;
  for (int c = lane; c < C; c += 32) {
    const float g = dr[c] * gamma[c];
    a += g;
    b += g * (xr[c] - mean) * rstd;
  }
  a = wsum(a) / C;
  b = wsum(b) / C;
  for (int c = lane; c < C; c += 32) {
    const float xh = (xr[c] - mean) * rstd;
    const float dx = rstd * (dr[c] * gamma[c] - a - xh * b);
    out[row * C + c] = (res ? res[row * C + c] : 0.f) + dx;
  }
  if (lane == 0 && stats != nullptr) stats[row] = make_float2(mean, rstd);
}
// Post-LN LayerNorm backward w.r.t. the input r = res + block output, warp per row, 4 consecutive channels per lane
// step: dy = dya + (dyb ? dyb : 0) (residual path + block path of the LayerNorm's output), out = dLN/dr(dy).  Also, for
// the block that feeds r: v = m * out with m the dropout mask of `site` (p = 0: no mask, v = out), written as fp32 to
// mout (optional) and as GEMM operand planes to op ([rows, planes * C], as split_rows writes them).  Stores (mean, rstd)
// per row for the parameter-gradient kernel.
__global__ void __launch_bounds__(256)
ln_post_bwd_dx_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ dya,
                      const float* __restrict__ dyb, float* __restrict__ out, float* __restrict__ mout,
                      __nv_bfloat16* __restrict__ op, int planes, float2* __restrict__ stats, long long rows, int C, float eps,
                      float p, const unsigned long long* __restrict__ seed, unsigned int site) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int C4 = C / 4;
  const float4* xr = reinterpret_cast<const float4*>(x + row * C);
  const float4* ar = reinterpret_cast<const float4*>(dya + row * C);
  const float4* br = dyb ? reinterpret_cast<const float4*>(dyb + row * C) : nullptr;
  const float4* g4 = reinterpret_cast<const float4*>(gamma);
  float s = 0.f;
  for (int c = lane; c < C4; c += 32) { const float4 v = xr[c]; s += (v.x + v.y) + (v.z + v.w); }
  const float mean = wsum(s) / C;
  float q = 0.f;
  for (int c = lane; c < C4; c += 32) {
    const float4 v = xr[c];
    const float d0 = v.x - mean, d1 = v.y - mean, d2 = v.z - mean, d3 = v.w - mean;
    q += (d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3);
  }
  const float rstd = rsqrtf(wsum(q) / C + eps);
  auto grad = [&](int c) {        // dy * gamma
    float4 d = ar[c];
    if (br) { const float4 e = br[c]; d.x += e.x; d.y += e.y; d.z += e.z; d.w += e.w; }
    const float4 g = g4[c];
    return make_float4(d.x * g.x, d.y * g.y, d.z * g.z, d.w * g.w);
  };
  float a = 0.f, b = 0.f;
  for (int c = lane; c < C4; c += 32) {
    const float4 g = grad(c), v = xr[c];
    a += (g.x + g.y) + (g.z + g.w);
    b += ((g.x * (v.x - mean) + g.y * (v.y - mean)) + (g.z * (v.z - mean) + g.w * (v.w - mean))) * rstd;
  }
  a = wsum(a) / C;
  b = wsum(b) / C;
  for (int c = lane; c < C4; c += 32) {
    const float4 g = grad(c), v = xr[c];
    float4 d;
    d.x = rstd * (g.x - a - (v.x - mean) * rstd * b);
    d.y = rstd * (g.y - a - (v.y - mean) * rstd * b);
    d.z = rstd * (g.z - a - (v.z - mean) * rstd * b);
    d.w = rstd * (g.w - a - (v.w - mean) * rstd * b);
    reinterpret_cast<float4*>(out + row * C)[c] = d;
    if (p > 0.f) {
      const float4 m = dropout_mask4(*seed, row * C4 + c, site, p);
      d = make_float4(m.x * d.x, m.y * d.y, m.z * d.z, m.w * d.w);
    }
    if (mout) reinterpret_cast<float4*>(mout + row * C)[c] = d;
    __nv_bfloat16* o = op + row * ((long long)planes * C) + 4 * c;
    const __nv_bfloat162 h0 = __floats2bfloat162_rn(d.x, d.y), h1 = __floats2bfloat162_rn(d.z, d.w);
    *reinterpret_cast<uint2*>(o) = make_uint2(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1));
    if (planes > 1) {
      const float2 f0 = __bfloat1622float2(h0), f1 = __bfloat1622float2(h1);
      *reinterpret_cast<uint2*>(o + C) = make_uint2(pack_bf16(d.x - f0.x, d.y - f0.y), pack_bf16(d.z - f1.x, d.w - f1.y));
    }
  }
  if (lane == 0) stats[row] = make_float2(mean, rstd);
}

// dgamma[c] = sum_r dy[r,c] xhat[r,c], dbeta[c] = sum_r dy[r,c]; SUM2: dy = dy + dy2 (the post-LN backward's two paths)
template <bool SUM2>
__global__ void __launch_bounds__(1024)
ln_bwd_params_kernel(const float* __restrict__ x, const float* __restrict__ dy, const float* __restrict__ dy2,
                     const float2* __restrict__ stats, long long rows, int C, float* __restrict__ dgamma, float* __restrict__ dbeta) {
  __shared__ float pg[CS_PH][33], pb[CS_PH][33];
  const int j = threadIdx.x % 32, ph = threadIdx.x / 32;
  const int c = blockIdx.x * 32 + j;
  float sg = 0.f, sb = 0.f;
  if (c < C)
    for (long long r = ph; r < rows; r += CS_PH) {
      const float2 st = stats[r];
      const float d = SUM2 ? dy[r * C + c] + dy2[r * C + c] : dy[r * C + c];
      sg += d * (x[r * C + c] - st.x) * st.y;
      sb += d;
    }
  pg[ph][j] = sg; pb[ph][j] = sb;
  __syncthreads();
  if (ph == 0 && c < C) {
    float tg = 0.f, tb = 0.f;
#pragma unroll
    for (int k = 0; k < CS_PH; ++k) { tg += pg[k][j]; tb += pb[k][j]; }
    dgamma[c] = tg; dbeta[c] = tb;
  }
}

// (A variant with two threads per row — 32 channels each in registers, 16-byte broadcast loads of the other side — measured
// slower: dq 303 vs 182 us, dk/dv 406 vs 268 us at 8 x 16 heads x 150 frames; this one-thread-per-row form is kept.)
// ---- attention backward.  Q, K, V, dO, O: [B*L, ld] matrices with the heads side by side (64 channels each), any float
// dtype; lse [B, H, L] = log-sum-exp of every query's scores (from the forward); key_pad [B, L] (1 = masked) or null.
// P_ij = exp(q_i . k_j - lse_i), D_i = dO_i . O_i, dS_ij = P_ij (dO_i . v_j - D_i);
// dQ_i = sum_j dS_ij k_j, dK_j = sum_i dS_ij q_i, dV_j = sum_i P_ij dO_i.
constexpr int AB_T = 32;       // queries (dq kernel) / keys (dkv kernel) per CTA
constexpr int AB_KT = 32;      // rows of the other side per shared-memory tile
constexpr int AB_HD = 64;

__global__ void __launch_bounds__(256)
attention_bwd_dq_kernel(const void* __restrict__ Q, long long ldq, const void* __restrict__ K, long long ldk,
                        const void* __restrict__ V, long long ldv, int dt, const void* __restrict__ dO, const void* __restrict__ O,
                        long long ldo, int o_dt, const float* __restrict__ lse, const unsigned char* __restrict__ key_pad,
                        void* __restrict__ dQ, long long lddq, int dq_dt, float* __restrict__ Dbuf, int L, int H) {
  __shared__ __align__(16) float Ks[AB_KT][AB_HD];
  __shared__ __align__(16) float Vs[AB_KT][AB_HD];
  __shared__ unsigned char dead[AB_KT];
  __shared__ float Qs[AB_T][AB_HD + 1];        // this CTA's queries and their dO rows: thread = row, padded -> conflict-free
  __shared__ float Gs[AB_T][AB_HD + 1];
  const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * AB_T;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int qi = q0 + lane;
  const bool ok = qi < L;
  attn_load_tile<AB_T, AB_HD + 1, 256>(Q, dt, ldq, (long long)b * L, q0, L, h * AB_HD, &Qs[0][0]);
  attn_load_tile<AB_T, AB_HD + 1, 256>(dO, o_dt, ldo, (long long)b * L, q0, L, h * AB_HD, &Gs[0][0]);
  __syncthreads();
  float acc[AB_HD];
  float D = 0.f;
  {
    const long long qrow = (long long)b * L + (ok ? qi : 0);
#pragma unroll 8
    for (int d = 0; d < AB_HD; ++d) {
      const float o = ok ? ldb(O, o_dt, qrow * ldo + h * AB_HD + d) : 0.f;
      D = fmaf(Gs[lane][d], o, D);
    }
  }
#pragma unroll
  for (int d = 0; d < AB_HD; ++d) acc[d] = 0.f;
  const float my_lse = ok ? lse[((long long)b * H + h) * L + qi] : INFINITY;
  if (w == 0 && ok) Dbuf[((long long)b * H + h) * L + qi] = D;
  for (int k0 = 0; k0 < L; k0 += AB_KT) {
    __syncthreads();
    attn_load_tile<AB_KT, AB_HD, 256>(K, dt, ldk, (long long)b * L, k0, L, h * AB_HD, &Ks[0][0]);
    attn_load_tile<AB_KT, AB_HD, 256>(V, dt, ldv, (long long)b * L, k0, L, h * AB_HD, &Vs[0][0]);
    if (threadIdx.x < AB_KT) {
      const int key = k0 + threadIdx.x;
      dead[threadIdx.x] = (key >= L || (key_pad != nullptr && key_pad[(long long)b * L + key] != 0)) ? 1 : 0;
    }
    __syncthreads();
#pragma unroll 1
    for (int j = 0; j < AB_KT / 8; ++j) {
      const int r = w + 8 * j;
      if (dead[r]) continue;
      float s = 0.f, dp = 0.f;
#pragma unroll
      for (int d = 0; d < AB_HD; ++d) {
        s = fmaf(Qs[lane][d], Ks[r][d], s);
        dp = fmaf(Gs[lane][d], Vs[r][d], dp);
      }
      const float ds = __expf(s - my_lse) * (dp - D);
#pragma unroll
      for (int d = 0; d < AB_HD; ++d) acc[d] = fmaf(ds, Ks[r][d], acc[d]);
    }
  }
  float (*Acc)[AB_HD + 1] = Gs;          // dO rows are no longer needed
  // sum the 8 per-warp partials of every query in warp order
  for (int turn = 0; turn < 8; ++turn) {
    __syncthreads();
    if (w == turn) {
#pragma unroll
      for (int d = 0; d < AB_HD; ++d) Acc[lane][d] = (turn == 0 ? 0.f : Acc[lane][d]) + acc[d];
    }
  }
  __syncthreads();
  for (int e = threadIdx.x; e < AB_T * AB_HD; e += 256) {
    const int r = e / AB_HD, d = e % AB_HD;
    if (q0 + r < L) stb(dQ, dq_dt, ((long long)b * L + q0 + r) * lddq + h * AB_HD + d, Acc[r][d]);
  }
}

__global__ void __launch_bounds__(256)
attention_bwd_dkv_kernel(const void* __restrict__ Q, long long ldq, const void* __restrict__ K, long long ldk,
                         const void* __restrict__ V, long long ldv, int dt, const void* __restrict__ dO, long long ldo, int o_dt,
                         const float* __restrict__ lse, const float* __restrict__ Dbuf, const unsigned char* __restrict__ key_pad,
                         void* __restrict__ dK, void* __restrict__ dV, long long lddk, int dk_dt, int L, int H) {
  __shared__ float Ks[AB_T][AB_HD + 1];        // this CTA's keys / values: row = lane -> padded rows, conflict-free
  __shared__ float Vs[AB_T][AB_HD + 1];
  __shared__ __align__(16) float Qs[AB_KT][AB_HD];      // query tile: broadcast reads
  __shared__ __align__(16) float Gs[AB_KT][AB_HD];      // dO tile
  __shared__ float Ls[AB_KT], Ds[AB_KT];
  const int b = blockIdx.z, h = blockIdx.y, j0 = blockIdx.x * AB_T;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int kj = j0 + lane;
  const bool live = kj < L && !(key_pad != nullptr && key_pad[(long long)b * L + kj] != 0);
  attn_load_tile<AB_T, AB_HD + 1, 256>(K, dt, ldk, (long long)b * L, j0, L, h * AB_HD, &Ks[0][0]);
  attn_load_tile<AB_T, AB_HD + 1, 256>(V, dt, ldv, (long long)b * L, j0, L, h * AB_HD, &Vs[0][0]);
  float dk[AB_HD], dv[AB_HD];
#pragma unroll
  for (int d = 0; d < AB_HD; ++d) { dk[d] = 0.f; dv[d] = 0.f; }
  for (int i0 = 0; i0 < L; i0 += AB_KT) {
    __syncthreads();
    attn_load_tile<AB_KT, AB_HD, 256>(Q, dt, ldq, (long long)b * L, i0, L, h * AB_HD, &Qs[0][0]);
    attn_load_tile<AB_KT, AB_HD, 256>(dO, o_dt, ldo, (long long)b * L, i0, L, h * AB_HD, &Gs[0][0]);
    if (threadIdx.x < AB_KT) {
      const int qi = i0 + threadIdx.x;
      Ls[threadIdx.x] = qi < L ? lse[((long long)b * H + h) * L + qi] : INFINITY;     // exp(s - inf) = 0: no contribution
      Ds[threadIdx.x] = qi < L ? Dbuf[((long long)b * H + h) * L + qi] : 0.f;
    }
    __syncthreads();
    if (live) {
#pragma unroll 1
      for (int j = 0; j < AB_KT / 8; ++j) {
        const int r = w + 8 * j;
        float s = 0.f, dp = 0.f;
#pragma unroll
        for (int d = 0; d < AB_HD; ++d) {
          s = fmaf(Qs[r][d], Ks[lane][d], s);
          dp = fmaf(Gs[r][d], Vs[lane][d], dp);
        }
        const float p = __expf(s - Ls[r]);
        const float ds = p * (dp - Ds[r]);
#pragma unroll
        for (int d = 0; d < AB_HD; ++d) {
          dv[d] = fmaf(p, Gs[r][d], dv[d]);
          dk[d] = fmaf(ds, Qs[r][d], dk[d]);
        }
      }
    }
  }
  // merge the 8 per-warp partials in warp order (Qs / Gs are free now)
  float (*A1)[AB_HD + 1] = Ks;      // reuse: keys / values are no longer needed after the loop
  float (*A2)[AB_HD + 1] = Vs;
  for (int turn = 0; turn < 8; ++turn) {
    __syncthreads();
    if (w == turn) {
#pragma unroll
      for (int d = 0; d < AB_HD; ++d) {
        A1[lane][d] = (turn == 0 ? 0.f : A1[lane][d]) + dk[d];
        A2[lane][d] = (turn == 0 ? 0.f : A2[lane][d]) + dv[d];
      }
    }
  }
  __syncthreads();
  for (int e = threadIdx.x; e < AB_T * AB_HD; e += 256) {
    const int r = e / AB_HD, d = e % AB_HD;
    if (j0 + r >= L) continue;
    const long long o = ((long long)b * L + j0 + r) * lddk + h * AB_HD + d;
    stb(dK, dk_dt, o, A1[r][d]);
    stb(dV, dk_dt, o, A2[r][d]);
  }
}

__global__ void __launch_bounds__(256) scale_kernel(float* __restrict__ p, long long n, float s) {
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) p[i] *= s;
}

// positional-conv weight gradient, operand of one group: XS[(k * cg + i), p * kp + r] = XT[(g * cg + i), p * kp + r + k - KT/2]
// (zero outside [0, kp)): the K-major "im2col" of the transposed zero-gapped input, one row per (tap, input channel)
__global__ void __launch_bounds__(256)
posconv_shift_kernel(const __nv_bfloat16* __restrict__ XT, __nv_bfloat16* __restrict__ XS, int g, int cg, int KT, int planes,
                     long long kp) {
  const int row = blockIdx.y;                  // k * cg + i
  const int k = row / cg, i = row % cg;
  const long long shift = k - KT / 2;
  const __nv_bfloat16* src = XT + (long long)(g * cg + i) * planes * kp;
  __nv_bfloat16* dst = XS + (long long)row * planes * kp;
  for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < planes * kp; e += (long long)gridDim.x * 256) {
    const long long p = e / kp, r = e % kp;
    const long long rs = r + shift;
    dst[e] = (rs >= 0 && rs < kp) ? src[p * kp + rs] : __float2bfloat16_rn(0.f);
  }
}

// weight-norm backward of the positional conv (w = g v / ||v||, norm over (out, in) per tap: weight_norm(dim=2)).
// dw [D, KT, cg] = gradient w.r.t. the effective weight (o, tap, in) as the group GEMMs wrote it; v [D, cg, KT], g [KT].
// One CTA per tap: n_k = ||v_k||, dg_k = sum dw v / n_k.
__global__ void __launch_bounds__(256)
posconv_dg_kernel(const float* __restrict__ dw, const float* __restrict__ v, int D, int cg, int KT, float* __restrict__ dg,
                  float* __restrict__ norms) {
  const int k = blockIdx.x;
  double sq = 0.0, dot = 0.0;
  for (int e = threadIdx.x; e < D * cg; e += 256) {
    const int o = e / cg, i = e % cg;
    const float vv = v[((long long)o * cg + i) * KT + k];
    sq += (double)vv * vv;
    dot += (double)dw[((long long)o * KT + k) * cg + i] * vv;
  }
  __shared__ double s1[256], s2[256];
  s1[threadIdx.x] = sq; s2[threadIdx.x] = dot;
  __syncthreads();
  for (int t = 128; t > 0; t >>= 1) {
    if (threadIdx.x < t) { s1[threadIdx.x] += s1[threadIdx.x + t]; s2[threadIdx.x] += s2[threadIdx.x + t]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const double n = sqrt(s1[0]);
    norms[k] = (float)n;
    dg[k] = (float)(s2[0] / n);
  }
}
// dv[o,i,k] = (g_k / n_k) (dw[o,k,i] - v[o,i,k] dg_k / n_k)
__global__ void __launch_bounds__(256)
posconv_dv_kernel(const float* __restrict__ dw, const float* __restrict__ v, const float* __restrict__ g,
                  const float* __restrict__ dg, const float* __restrict__ norms, int D, int cg, int KT, float* __restrict__ dv) {
  const long long n = (long long)D * cg * KT;
  for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < n; e += (long long)gridDim.x * 256) {
    const int k = (int)(e % KT);
    const long long oi = e / KT;
    const int i = (int)(oi % cg);
    const long long o = oi / cg;
    const float nk = norms[k];
    dv[e] = (g[k] / nk) * (dw[(o * KT + k) * cg + i] - v[e] * dg[k] / nk);
  }
}

}  // namespace

int launch_scale(float* p, long long n, float s, cudaStream_t stream) {
  if (n <= 0) return 0;
  const long long blocks = (n + 1023) / 1024;
  scale_kernel<<<(unsigned)(blocks < 1184 ? blocks : 1184), 256, 0, stream>>>(p, n, s);
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_posconv_shift(const void* XT, void* XS, int g, int cg, int KT, int planes, long long kp, cudaStream_t stream) {
  dim3 grid((unsigned)((planes * kp + 256 * 8 - 1) / (256 * 8)), (unsigned)(KT * cg));
  posconv_shift_kernel<<<grid, 256, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(XT), reinterpret_cast<__nv_bfloat16*>(XS),
                                                 g, cg, KT, planes, kp);
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_posconv_weightnorm_bwd(const float* dw, const float* v, const float* g, int D, int cg, int KT, float* dg, float* dv,
                                  float* norms, cudaStream_t stream) {
  posconv_dg_kernel<<<KT, 256, 0, stream>>>(dw, v, D, cg, KT, dg, norms);
  AVH_CUDA_OK(cudaGetLastError());
  const long long n = (long long)D * cg * KT;
  const long long blocks = (n + 1023) / 1024;
  posconv_dv_kernel<<<(unsigned)(blocks < 4736 ? blocks : 4736), 256, 0, stream>>>(dw, v, g, dg, norms, D, cg, KT, dv);
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(2);
  return 0;
}

int launch_transpose_split(const void* in, int dt, long long ld, long long rows, int C, void* out, int planes, long long kpad,
                           float scale, cudaStream_t stream, int T, int Tp, long long out_ld) {
  AVH_CHECK(kpad % 64 == 0 && (T > 0 ? kpad >= rows / T * Tp : kpad >= rows),
            "transpose_split: K padding must cover the rows and be a multiple of 64");
  if (C <= 0) return 0;
  {
    const long long old_ = out_ld > 0 ? out_ld : (long long)planes * kpad;
    if (planes == 1 && scale == 1.0f && T == 0 && (dt == DT_BF16 || dt == DT_F32) && C % 8 == 0 && ld % 8 == 0 && old_ % 8 == 0 &&
        (reinterpret_cast<uintptr_t>(in) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0)
      return launch_transposeT(in, dt, ld, rows, C, out, kpad, old_, stream);       // 64 x 64 tiles, 16-byte accesses
  }
  dim3 grid((unsigned)((kpad + 31) / 32), (unsigned)((C + 31) / 32));
  transpose_split_kernel<<<grid, 256, 0, stream>>>(in, dt, ld, rows, C, reinterpret_cast<__nv_bfloat16*>(out), planes, kpad, scale,
                                                   T, Tp, out_ld > 0 ? out_ld : (long long)planes * kpad);
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_colsum(const void* in, int dt, long long ld, long long rows, int C, float* out, float scale, cudaStream_t stream) {
  if (C <= 0) return 0;
  colsum_kernel<<<(C + 31) / 32, 1024, 0, stream>>>(in, dt, ld, rows, C, out, scale);
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_gelu_fwd(const void* u, int u_dt, const float* res, void* out, int out_dt, long long n, cudaStream_t stream) {
  if (n <= 0) return 0;
  const long long blocks = (n + 256 * 4 - 1) / (256 * 4);
  gelu_fwd_kernel<<<(unsigned)(blocks < 4736 ? blocks : 4736), 256, 0, stream>>>(u, u_dt, res, out, out_dt, n);
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_gelu_bwd(const void* u, int u_dt, const void* dg, int dg_dt, void* du, int du_dt, long long n, cudaStream_t stream) {
  if (n <= 0) return 0;
  const long long blocks = (n + 256 * 4 - 1) / (256 * 4);
  gelu_bwd_kernel<<<(unsigned)(blocks < 4736 ? blocks : 4736), 256, 0, stream>>>(u, u_dt, dg, dg_dt, du, du_dt, n);
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_ln_bwd(const float* x, const float* gamma, const float* dy, const float* res, float* dx_out, float2* stats,
                  float* dgamma, float* dbeta, long long rows, int C, float eps, cudaStream_t stream) {
  if (rows <= 0) return 0;
  AVH_CHECK(stats != nullptr, "ln_bwd needs the per-row statistics buffer");
  ln_bwd_dx_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, stream>>>(x, gamma, dy, res, dx_out, stats, rows, C, eps);
  AVH_CUDA_OK(cudaGetLastError());
  ln_bwd_params_kernel<false><<<(C + 31) / 32, 1024, 0, stream>>>(x, dy, nullptr, stats, rows, C, dgamma, dbeta);
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(2);
  return 0;
}

int launch_ln_post_bwd(const float* x, const float* gamma, const float* dya, const float* dyb, float* dx_out, float* mout,
                       void* op, int planes, float2* stats, float* dgamma, float* dbeta, long long rows, int C, float eps,
                       float p, const unsigned long long* seed, unsigned int site, cudaStream_t stream) {
  if (rows <= 0) return 0;
  AVH_CHECK(stats != nullptr && op != nullptr, "ln_post_bwd needs the per-row statistics buffer and the operand output");
  AVH_CHECK(C % 4 == 0, "ln_post_bwd: row width must be a multiple of 4");
  AVH_CHECK(p == 0.f || (p > 0.f && p < 1.f && seed != nullptr), "ln_post_bwd: dropout probability in [0, 1), seed for p > 0");
  AVH_CHECK(dx_out != dya && dx_out != dyb && (mout == nullptr || (mout != dya && mout != dyb)),
            "ln_post_bwd: the outputs must not alias the incoming gradients (the parameter pass re-reads them)");
  ln_post_bwd_dx_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, stream>>>(x, gamma, dya, dyb, dx_out, mout,
                                                                        reinterpret_cast<__nv_bfloat16*>(op), planes, stats,
                                                                        rows, C, eps, p, seed, site);
  AVH_CUDA_OK(cudaGetLastError());
  if (dyb != nullptr)
    ln_bwd_params_kernel<true><<<(C + 31) / 32, 1024, 0, stream>>>(x, dya, dyb, stats, rows, C, dgamma, dbeta);
  else
    ln_bwd_params_kernel<false><<<(C + 31) / 32, 1024, 0, stream>>>(x, dya, nullptr, stats, rows, C, dgamma, dbeta);
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(2);
  return 0;
}

int launch_attention_bwd(const void* Q, long long ldq, const void* K, long long ldk, const void* V, long long ldv, int dt,
                         const void* dO, const void* O, long long ldo, int o_dt, const float* lse, const unsigned char* key_pad,
                         void* dQ, void* dK, void* dV, long long ldd, int d_dt, float* Dbuf, int B, int H, int L,
                         cudaStream_t stream) {
  AVH_CHECK(B > 0 && H > 0 && L > 0 && B <= 65535 && H <= 65535, "bad attention shape");
  dim3 grid((L + AB_T - 1) / AB_T, H, B);
  attention_bwd_dq_kernel<<<grid, 256, 0, stream>>>(Q, ldq, K, ldk, V, ldv, dt, dO, O, ldo, o_dt, lse, key_pad, dQ, ldd, d_dt,
                                                    Dbuf, L, H);
  AVH_CUDA_OK(cudaGetLastError());
  attention_bwd_dkv_kernel<<<grid, 256, 0, stream>>>(Q, ldq, K, ldk, V, ldv, dt, dO, ldo, o_dt, lse, Dbuf, key_pad, dK, dV, ldd,
                                                     d_dt, L, H);
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(2);
  return 0;
}

}  // namespace avh
