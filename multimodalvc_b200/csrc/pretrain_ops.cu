// Pretraining-mode extras of AV-HuBERT (SURVEY 8(f) rank 4): the device side of span masking and the masked-prediction
// logits and their backward.  None of this is on the benchmarked step; the kernels are HBM-bound copies / small fp32
// contractions.
//
//  * apply_input_mask (avhubert/hubert.py:442-494) and apply_feature_mask (:496-536): the host draws the spans
//    (masking.py, numpy RNG in the reference's order) and turns them into ONE int32 code per (clip, frame):
//      code >= 0  : take frame `code` (= b' * T + t') of the INPUT tensor   (same_other_seq / same_seq substitution)
//      code == -1 : keep the clip's own frame
//      code == -2 : zeros                                                   (B == 1, hubert.py:465-466)
//      code == -3 : the mask embedding                                      (audio / feature masking, :467-468, :511)
//    The reference gathers its right-hand side before it assigns, so every source is read from the un-substituted
//    tensor: one out-of-place pass.  Two layouts: contiguous units (video frames [B,1,T,H*W], token rows [B,T,C],
//    optionally with a per-(clip, channel) zero mask = mask_channel_prob, :517-534) and the collater's strided audio
//    [B,C,T].
//  * compute_logits (hubert.py:576-589): logits[m,v] = <f_m, e_v> / temp  ('dot') or
//    <f_m, e_v> / max(|f_m| |e_v|, 1e-6) / temp ('cosine'), fp32 throughout; with a bias and no scaling the same kernel
//    is final_proj (nn.Linear, hubert.py:654).
//  * features_pen (hubert.py:629): mean of squares, float64 partial sums.
//  * the backward of compute_logits / final_proj for the training-mode pretraining step: fp32 row norms, the cosine
//    chain rule's row / column sums, the contractions dF = G E and dE = G^T F (64 x 64 tiles, split over the long axis
//    with partials added in order), the column sums of dbias; no atomics, so a step replays bit for bit.  The pen
//    gradient of the fused features (2 dL/dpen / numel) fused, dL/dpen read from the plan's device word.
#include "common.cuh"
#include "kernels.h"

#include <cuda_fp16.h>

#include <algorithm>

namespace avh {
namespace {

__device__ __forceinline__ float ldv(const void* p, int dt, long long i) {
  if (dt == DT_BF16) return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[i]);
  if (dt == DT_F16) return __half2float(reinterpret_cast<const __half*>(p)[i]);
  return reinterpret_cast<const float*>(p)[i];
}
__device__ __forceinline__ void stv(void* out, int dt, long long i, float v) {
  if (dt == DT_BF16) reinterpret_cast<__nv_bfloat16*>(out)[i] = __float2bfloat16_rn(v);
  else if (dt == DT_F16) reinterpret_cast<__half*>(out)[i] = __float2half_rn(v);
  else reinterpret_cast<float*>(out)[i] = v;
}

// contiguous units of U elements: out unit u = in unit code[u] | own | zeros | emb
// 16-byte vectors when the unit size allows (video frames: 7744 elements; token rows: C % 8 == 0)
template <int VEC>
__global__ void __launch_bounds__(256)
mask_units_kernel(const unsigned char* __restrict__ in, unsigned char* __restrict__ out, const int* __restrict__ code,
                  const void* __restrict__ emb, int emb_dt, int dt, long long units, long long unit_bytes, int U,
                  const unsigned char* __restrict__ chan_zero, int T) {
  const long long u = blockIdx.x;
  if (u >= units) return;
  const int cd = code[u];
  const unsigned char* src = in + (cd >= 0 ? (long long)cd : u) * unit_bytes;
  unsigned char* dst = out + u * unit_bytes;
  const unsigned char* cz = chan_zero ? chan_zero + (u / T) * (long long)U : nullptr;
  if (cd == -3 || cz != nullptr || VEC == 1) {
    for (int i = threadIdx.x; i < U; i += blockDim.x) {
      float v;
      if (cd == -3) v = ldv(emb, emb_dt, i);
      else if (cd == -2) v = 0.f;
      else v = ldv(src, dt, i);
      if (cz != nullptr && cz[i]) v = 0.f;
      stv(dst, dt, i, v);
    }
    return;
  }
  const int nvec = (int)(unit_bytes / 16);
  const uint4* s4 = reinterpret_cast<const uint4*>(src);
  uint4* d4 = reinterpret_cast<uint4*>(dst);
  for (int i = threadIdx.x; i < nvec; i += blockDim.x) d4[i] = cd == -2 ? make_uint4(0, 0, 0, 0) : s4[i];
}

// strided audio [B,C,T] -> contiguous [B,C,T]; a 32 (channels) x 32 (frames) tile per CTA, reads follow the input's
// fastest stride through a transposing smem tile when the view is the collater's (time-major storage)
__global__ void __launch_bounds__(256)
mask_bct_kernel(const void* __restrict__ in, int dt, long long sb, long long sc, long long st, void* __restrict__ out,
                int out_dt, const int* __restrict__ code, const void* __restrict__ emb, int emb_dt, int B, int C, int T) {
  __shared__ float tile[32][33];
  __shared__ int cds[32];
  const int b = blockIdx.z, c0 = blockIdx.y * 32, t0 = blockIdx.x * 32;
  if (threadIdx.x < 32) cds[threadIdx.x] = t0 + threadIdx.x < T ? code[(long long)b * T + t0 + threadIdx.x] : -1;
  __syncthreads();
  const bool time_major = sc < st;                  // channels contiguous in memory: walk channels fastest on the read
  for (int k = threadIdx.x; k < 1024; k += 256) {
    const int i = time_major ? k % 32 : k / 32;     // channel within the tile
    const int j = time_major ? k / 32 : k % 32;     // frame within the tile
    const int c = c0 + i, t = t0 + j;
    if (c >= C || t >= T) continue;
    const int cd = cds[j];
    float v;
    if (cd == -3) v = ldv(emb, emb_dt, c);
    else if (cd == -2) v = 0.f;
    else {
      const long long sbb = cd >= 0 ? cd / T : b, stt = cd >= 0 ? cd % T : t;
      v = ldv(in, dt, sbb * sb + (long long)c * sc + stt * st);
    }
    tile[i][j] = v;
  }
  __syncthreads();
  for (int k = threadIdx.x; k < 1024; k += 256) {
    const int i = k / 32, j = k % 32;
    const int c = c0 + i, t = t0 + j;
    if (c < C && t < T) stv(out, out_dt, ((long long)b * C + c) * T + t, tile[i][j]);
  }
}

// out[m, v] = (sum_k f[m,k] e[v,k] + bias[v]) * scale(m, v): 64 x 64 tile, 16-wide k slices, 4 x 4 per thread, fp32 FMA.
// mode 0: scale = inv_temp; mode 1 (cosine): scale = inv_temp / max(|f_m| |e_v|, 1e-6), the norms accumulated from the
// same smem slices
__global__ void __launch_bounds__(256)
logits_kernel(const void* __restrict__ F, int f_dt, long long ldf, const void* __restrict__ E, int e_dt, long long lde,
              const float* __restrict__ bias, float* __restrict__ out, long long ldo, long long M, int V, int K, int mode,
              float inv_temp) {
  __shared__ float fs[16][65], es[16][65];
  __shared__ float fn[64], en[64];
  const long long m0 = (long long)blockIdx.y * 64;
  const int v0 = blockIdx.x * 64;
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
  float acc[4][4] = {};
  float nrm = 0.f;                                  // threads 0..63: |f|^2 of row tid; 64..127: |e|^2 of column tid-64
  for (int k0 = 0; k0 < K; k0 += 16) {
    for (int q = threadIdx.x; q < 1024; q += 256) {
      const int r = q / 16, kk = q % 16;
      const int k = k0 + kk;
      fs[kk][r] = (m0 + r < M && k < K) ? ldv(F, f_dt, (m0 + r) * ldf + k) : 0.f;
      es[kk][r] = (v0 + r < V && k < K) ? ldv(E, e_dt, (long long)(v0 + r) * lde + k) : 0.f;
    }
    __syncthreads();
    if (mode == 1 && threadIdx.x < 128) {
      const int r = threadIdx.x % 64;
#pragma unroll
      for (int kk = 0; kk < 16; ++kk) {
        const float x = threadIdx.x < 64 ? fs[kk][r] : es[kk][r];
        nrm = fmaf(x, x, nrm);
      }
    }
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = fs[kk][ty * 4 + i]; b[i] = es[kk][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
  if (mode == 1) {
    if (threadIdx.x < 64) fn[threadIdx.x] = sqrtf(nrm);
    else if (threadIdx.x < 128) en[threadIdx.x - 64] = sqrtf(nrm);
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int v = v0 + tx * 4 + j;
      if (v >= V) continue;
      float x = acc[i][j] + (bias ? bias[v] : 0.f);
      if (mode == 1) x = x / fmaxf(fn[ty * 4 + i] * en[tx * 4 + j], 1e-6f);
      out[m * ldo + v] = x * inv_temp;
    }
  }
}

// ---- backward of logits_kernel.  With s = <f_m, e_v> + bias[v] and out = s * scale(m, v):
//   G[m,v] = dout[m,v] * scale(m,v)                                    (gradient of s)
//   cosine, where |f_m| |e_v| >= 1e-6 (torch.clamp passes the gradient there, the clamped denominator is a constant):
//   d den = -dout * out / den, den = |f_m| |e_v|, so d f_m += f_m * (-sum_v dout*out) / |f_m|^2 and likewise for e_v.
//   dF = G E + c_f * F,  dE = G^T F + c_e * E,  dbias = column sums of G.
// Every reduction runs in a fixed order (no atomics): a step replays bit for bit.

// |x_r| of every row, a warp per row
__global__ void __launch_bounds__(256)
row_norms_kernel(const void* __restrict__ X, int dt, long long ld, long long rows, int K, float* __restrict__ out) {
  const long long r = (long long)blockIdx.x * 8 + threadIdx.x / 32;
  if (r >= rows) return;
  const int lane = threadIdx.x & 31;
  float s = 0.f;
  for (int k = lane; k < K; k += 32) {
    const float x = ldv(X, dt, r * ld + k);
    s = fmaf(x, x, s);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) out[r] = sqrtf(s);
}

// cosine: rs[m] = sum over the unclamped v of dout * out, a warp per row
__global__ void __launch_bounds__(256)
logits_rowsum_kernel(const float* __restrict__ dout, const float* __restrict__ lg, long long ldo, const float* __restrict__ fn,
                     const float* __restrict__ en, long long M, int V, float* __restrict__ rs) {
  const long long m = (long long)blockIdx.x * 8 + threadIdx.x / 32;
  if (m >= M) return;
  const int lane = threadIdx.x & 31;
  const float f = fn[m];
  float s = 0.f;
  for (int v = lane; v < V; v += 32)
    if (f * en[v] >= 1e-6f) s = fmaf(dout[m * ldo + v], lg[m * ldo + v], s);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) rs[m] = s;
}

// column sums over m: cs[v] = sum of dout * out over the unclamped m (cosine), db[v] = sum of G[m, v] (either may be null);
// 32 columns x 8 row phases per block, the phases added in order
__global__ void __launch_bounds__(256)
logits_colsum_kernel(const float* __restrict__ dout, const float* __restrict__ lg, long long ldo, const float* __restrict__ fn,
                     const float* __restrict__ en, long long M, int V, int mode, float inv_temp, float* __restrict__ cs,
                     float* __restrict__ db) {
  __shared__ float sq[8][33], sg[8][33];
  const int lane = threadIdx.x & 31, ph = threadIdx.x / 32;
  const int v = blockIdx.x * 32 + lane;
  float a = 0.f, g = 0.f;
  if (v < V) {
    const float e = mode == 1 ? en[v] : 0.f;
    for (long long m = ph; m < M; m += 8) {
      const float d = dout[m * ldo + v];
      if (mode == 1) {
        const float den = fn[m] * e;
        if (den >= 1e-6f) a = fmaf(d, lg[m * ldo + v], a);
        g = fmaf(d, inv_temp / fmaxf(den, 1e-6f), g);
      } else {
        g = fmaf(d, inv_temp, g);
      }
    }
  }
  sq[ph][lane] = a;
  sg[ph][lane] = g;
  __syncthreads();
  if (ph == 0 && v < V) {
    float ta = 0.f, tg = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { ta += sq[i][lane]; tg += sg[i][lane]; }
    if (cs != nullptr) cs[v] = ta;
    if (db != nullptr) db[v] = tg;
  }
}

// out[r, k] = sum_j G(r, j) X[j, k] (+ c_r Y[r, k], cosine): TR = false: r = m, j = v (dF, X = E, Y = F);
// TR = true: r = v, j = m (dE, X = F, Y = E).  64 x 64 tile, 16-wide j slices, G formed while its tile is loaded.
// Split j (few output tiles, long j: the weight-like gradients): block z sums j in [z jchunk, (z+1) jchunk) into
// partial [gridDim.z, R, K], which logits_grad_reduce_kernel adds up in z order.
template <bool TR>
__global__ void __launch_bounds__(256)
logits_grad_kernel(const float* __restrict__ dout, long long ldo, const float* __restrict__ fn, const float* __restrict__ en,
                   long long M, int V, int K, int mode, float inv_temp, const void* __restrict__ X, int x_dt, long long ldx,
                   const void* __restrict__ Y, int y_dt, long long ldy, const float* __restrict__ rsum, float* __restrict__ out,
                   long long ldd, long long jchunk, float* __restrict__ partial) {
  __shared__ float gs[16][65], xs[16][65];
  const long long R = TR ? (long long)V : M;
  const long long jb = (long long)blockIdx.z * jchunk;
  const long long J = min(TR ? M : (long long)V, jb + jchunk);
  const long long r0 = (long long)blockIdx.y * 64;
  const int k0 = blockIdx.x * 64;
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
  float acc[4][4] = {};
  for (long long j0 = jb; j0 < J; j0 += 16) {
    for (int q = threadIdx.x; q < 1024; q += 256) {
      const int rr = TR ? q % 64 : q / 16, jj = TR ? q / 64 : q % 16;     // reads of dout follow its contiguous axis
      const long long r = r0 + rr, j = j0 + jj;
      float g = 0.f;
      if (r < R && j < J) {
        const long long m = TR ? j : r, v = TR ? r : j;
        g = dout[m * ldo + v] * (mode == 1 ? inv_temp / fmaxf(fn[m] * en[v], 1e-6f) : inv_temp);
      }
      gs[jj][rr] = g;
      const int kk = q % 64, jx = q / 64;
      xs[jx][kk] = (j0 + jx < J && k0 + kk < K) ? ldv(X, x_dt, (j0 + jx) * ldx + k0 + kk) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int jj = 0; jj < 16; ++jj) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = gs[jj][ty * 4 + i]; b[i] = xs[jj][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long r = r0 + ty * 4 + i;
    if (r >= R) continue;
    if (partial != nullptr) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int k = k0 + tx * 4 + j;
        if (k < K) partial[((long long)blockIdx.z * R + r) * K + k] = acc[i][j];
      }
      continue;
    }
    float c = 0.f;
    if (mode == 1 && rsum[r] != 0.f) {                // a row whose every pair is clamped has rsum 0 (and maybe norm 0)
      const float n = TR ? en[r] : fn[r];
      c = -rsum[r] / (n * n);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + tx * 4 + j;
      if (k >= K) continue;
      float v = acc[i][j];
      if (c != 0.f) v = fmaf(c, ldv(Y, y_dt, r * ldy + k), v);
      out[r * ldd + k] = v;
    }
  }
}

template <bool TR>
__global__ void __launch_bounds__(256)
logits_grad_reduce_kernel(const float* __restrict__ partial, int splits, long long R, int K, int mode, const float* __restrict__ fn,
                          const float* __restrict__ en, const void* __restrict__ Y, int y_dt, long long ldy,
                          const float* __restrict__ rsum, float* __restrict__ out, long long ldd) {
  const long long n = R * K;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const long long r = i / K;
    const int k = (int)(i % K);
    float v = 0.f;
    for (int z = 0; z < splits; ++z) v += partial[z * n + i];
    if (mode == 1 && rsum[r] != 0.f) {
      const float nr = TR ? en[r] : fn[r];
      v = fmaf(-rsum[r] / (nr * nr), ldv(Y, y_dt, r * ldy + k), v);
    }
    out[r * ldd + k] = v;
  }
}

// features_pen = mean(fused^2): d(fused) += (2 dL/dpen / numel) fused, dL/dpen read from a device word
__global__ void __launch_bounds__(256)
pen_grad_kernel(const float* __restrict__ x, float* __restrict__ dx, long long n, const float* __restrict__ dpen, float scale) {
  const float c = dpen[0] * scale;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) dx[i] = fmaf(c, x[i], dx[i]);
}

__global__ void __launch_bounds__(256)
sumsq_kernel(const void* __restrict__ x, int dt, long long n, double* __restrict__ acc) {
  double s = 0.0;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const double v = (double)ldv(x, dt, i);
    s += v * v;
  }
  __shared__ double sh[256];
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int k = 128; k > 0; k >>= 1) {
    if (threadIdx.x < k) sh[threadIdx.x] += sh[threadIdx.x + k];
    __syncthreads();
  }
  if (threadIdx.x == 0) atomicAdd(acc, sh[0]);
}

}  // namespace

int launch_mask_units(const void* in, void* out, int dt, const int* code, const void* emb, int emb_dt, long long units,
                      int U, const unsigned char* chan_zero, int T, cudaStream_t stream) {
  if (units <= 0) return 0;
  const long long unit_bytes = (long long)U * (dt == DT_F32 ? 4 : 2);
  const bool vec = unit_bytes % 16 == 0 && (reinterpret_cast<uintptr_t>(in) % 16 == 0) &&
                   (reinterpret_cast<uintptr_t>(out) % 16 == 0);
  AVH_CHECK(units <= 0x7fffffffLL, "too many units");
  if (vec)
    mask_units_kernel<4><<<(unsigned)units, 256, 0, stream>>>(
        reinterpret_cast<const unsigned char*>(in), reinterpret_cast<unsigned char*>(out), code, emb, emb_dt, dt, units,
        unit_bytes, U, chan_zero, T);
  else
    mask_units_kernel<1><<<(unsigned)units, 256, 0, stream>>>(
        reinterpret_cast<const unsigned char*>(in), reinterpret_cast<unsigned char*>(out), code, emb, emb_dt, dt, units,
        unit_bytes, U, chan_zero, T);
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_mask_bct(const void* in, int dt, long long sb, long long sc, long long st, void* out, int out_dt,
                    const int* code, const void* emb, int emb_dt, int B, int C, int T, cudaStream_t stream) {
  if (B <= 0 || C <= 0 || T <= 0) return 0;
  dim3 grid((T + 31) / 32, (C + 31) / 32, B);
  mask_bct_kernel<<<grid, 256, 0, stream>>>(in, dt, sb, sc, st, out, out_dt, code, emb, emb_dt, B, C, T);
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_logits(const void* F, int f_dt, long long ldf, const void* E, int e_dt, long long lde, const float* bias,
                  float* out, long long ldo, long long M, int V, int K, int mode, float inv_temp, cudaStream_t stream) {
  if (M <= 0 || V <= 0) return 0;
  dim3 grid((V + 63) / 64, (unsigned)((M + 63) / 64));
  logits_kernel<<<grid, 256, 0, stream>>>(F, f_dt, ldf, E, e_dt, lde, bias, out, ldo, M, V, K, mode, inv_temp);
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

// j splits of one contraction [R, K] over J: about two blocks per SM, each split at least 256 long (multiples of 16)
int logits_grad_splits(long long R, long long J, int K) {
  const long long tiles = ((R + 63) / 64) * ((K + 63) / 64);
  long long S = std::min<long long>((2 * 148 + tiles - 1) / tiles, J / 256);
  return (int)std::max<long long>(1, std::min<long long>(S, 32));
}

long long logits_bwd_scratch_floats(long long M, int V, int K) {
  const long long a = logits_grad_splits(M, V, K), b = logits_grad_splits(V, M, K);
  const long long pa = a > 1 ? a * M * K : 0, pb = b > 1 ? b * (long long)V * K : 0;
  return 2 * (M + V) + std::max(pa, pb);
}

int launch_logits_bwd(const void* F, int f_dt, long long ldf, const void* E, int e_dt, long long lde, long long M, int V, int K,
                      int mode, float inv_temp, const float* logits, const float* dlogits, long long ldo, float* dF, long long ldd_f,
                      float* dE, long long ldd_e, float* dbias, float* scratch, cudaStream_t stream) {
  if (M <= 0 || V <= 0) return 0;
  AVH_CHECK(M < (1ll << 31) / 64 && (long long)V < (1ll << 31) / 64, "too many rows");
  float *fn = nullptr, *en = nullptr, *rs = nullptr, *cs = nullptr;
  if (mode == 1) {        // scratch: |f| [M], |e| [V], row sums [M], column sums [V]
    fn = scratch; en = fn + M; rs = en + V; cs = rs + M;
    row_norms_kernel<<<(unsigned)((M + 7) / 8), 256, 0, stream>>>(F, f_dt, ldf, M, K, fn);
    row_norms_kernel<<<(unsigned)((V + 7) / 8), 256, 0, stream>>>(E, e_dt, lde, V, K, en);
    logits_rowsum_kernel<<<(unsigned)((M + 7) / 8), 256, 0, stream>>>(dlogits, logits, ldo, fn, en, M, V, rs);
    count_launch(3);
  }
  if (mode == 1 || dbias != nullptr) {
    logits_colsum_kernel<<<(unsigned)((V + 31) / 32), 256, 0, stream>>>(dlogits, logits, ldo, fn, en, M, V, mode, inv_temp,
                                                                         mode == 1 ? cs : nullptr, dbias);
    count_launch(1);
  }
  float* partial = scratch + 2 * (M + V);
  if (dF != nullptr) {
    const int S = logits_grad_splits(M, V, K);
    dim3 grid((K + 63) / 64, (unsigned)((M + 63) / 64), S);
    const long long jc = (V + S - 1) / S;
    logits_grad_kernel<false><<<grid, 256, 0, stream>>>(dlogits, ldo, fn, en, M, V, K, mode, inv_temp, E, e_dt, lde, F, f_dt, ldf,
                                                        rs, dF, ldd_f, jc, S > 1 ? partial : nullptr);
    if (S > 1)
      logits_grad_reduce_kernel<false><<<1184, 256, 0, stream>>>(partial, S, M, K, mode, fn, en, F, f_dt, ldf, rs, dF, ldd_f);
    count_launch(S > 1 ? 2 : 1);
  }
  if (dE != nullptr) {
    const int S = logits_grad_splits(V, M, K);
    dim3 grid((K + 63) / 64, (unsigned)((V + 63) / 64), S);
    const long long jc = (M + S - 1) / S;
    logits_grad_kernel<true><<<grid, 256, 0, stream>>>(dlogits, ldo, fn, en, M, V, K, mode, inv_temp, F, f_dt, ldf, E, e_dt, lde,
                                                       cs, dE, ldd_e, jc, S > 1 ? partial : nullptr);
    if (S > 1)
      logits_grad_reduce_kernel<true><<<1184, 256, 0, stream>>>(partial, S, V, K, mode, fn, en, E, e_dt, lde, cs, dE, ldd_e);
    count_launch(S > 1 ? 2 : 1);
  }
  AVH_CUDA_OK(cudaGetLastError());
  return 0;
}

int launch_pen_grad(const float* x, float* dx, long long n, const float* dpen, float scale, cudaStream_t stream) {
  if (n <= 0) return 0;
  const long long blocks = (n + 256 * 8 - 1) / (256 * 8);
  pen_grad_kernel<<<(unsigned)(blocks < 1184 ? blocks : 1184), 256, 0, stream>>>(x, dx, n, dpen, scale);
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_sumsq(const void* x, int dt, long long n, double* acc, cudaStream_t stream) {
  AVH_CUDA_OK(cudaMemsetAsync(acc, 0, sizeof(double), stream));
  if (n <= 0) return 0;
  const long long blocks = (n + 256 * 8 - 1) / (256 * 8);
  sumsq_kernel<<<(unsigned)(blocks < 1184 ? blocks : 1184), 256, 0, stream>>>(x, dt, n, acc);
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

}  // namespace avh
