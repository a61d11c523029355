// HBM/L2-bound helper kernels of the AV-HuBERT hot path: LayerNorm, layout changes, the explicit
// im2col gathers that feed the tcgen05 GEMM (round-1 lip frontend), pooling and precision splitting.
// All loads/stores are 16-byte vectors along the channel (innermost) dimension where the layout allows.
#include "common.cuh"
#include "kernels.h"

#include <cuda_fp16.h>

namespace avh {
namespace {

__device__ __forceinline__ float load_any(const void* p, int dt, long long i) {
  if (dt == DT_BF16) return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[i]);
  if (dt == DT_F16) return __half2float(reinterpret_cast<const __half*>(p)[i]);
  return reinterpret_cast<const float*>(p)[i];
}
__device__ __forceinline__ void store_lp(void* out, int dt, long long i, float v) {
  if (dt == DT_BF16) reinterpret_cast<__nv_bfloat16*>(out)[i] = __float2bfloat16_rn(v);
  else if (dt == DT_F16) reinterpret_cast<__half*>(out)[i] = __float2half_rn(v);
  else reinterpret_cast<float*>(out)[i] = v;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------------------------- LayerNorm
// one warp per row; two-pass mean/variance in fp32 (rows are <= 8 KB and stay in L1 between passes).
// Reference: torch.nn.LayerNorm via fairseq/fairseq/modules/layer_norm.py:51-56, eps 1e-5.
__global__ void layernorm_kernel(const void* __restrict__ in, int in_dt, long long ld_in,
                                 const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                 float* __restrict__ out_f32, void* __restrict__ out_lp, int lp_dt,
                                 const unsigned char* __restrict__ row_zero, long long rows, int C) {
  pdl_launch_dependents();
  pdl_wait();
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const long long base = row * ld_in;
  const bool zero = row_zero != nullptr && row_zero[row] != 0;
  float s = 0.f;
  for (int c = lane; c < C; c += 32) s += load_any(in, in_dt, base + c);
  const float mean = warp_sum(s) / (float)C;
  float q = 0.f;
  for (int c = lane; c < C; c += 32) {
    const float d = load_any(in, in_dt, base + c) - mean;
    q += d * d;
  }
  const float rstd = rsqrtf(warp_sum(q) / (float)C + eps);
  for (int c = lane; c < C; c += 32) {
    float v = (load_any(in, in_dt, base + c) - mean) * rstd;
    if (gamma != nullptr) v = v * gamma[c] + beta[c];
    if (zero) v = 0.f;
    if (out_f32 != nullptr) out_f32[row * C + c] = v;
    if (out_lp != nullptr) store_lp(out_lp, lp_dt, row * C + c, v);
  }
}

// fp32 rows with C % 128 == 0: float4 loads, row cached in registers (C <= 2048)
// IN_BF16: the row is bf16 (the fused audio|video features in bf16 mode) instead of fp32.
template <int VEC, bool IN_BF16 = false>
__global__ void layernorm_f32_vec_kernel(const float* __restrict__ in, long long ld_in,
                                         const float* __restrict__ gamma, const float* __restrict__ beta,
                                         float eps, float* __restrict__ out_f32, void* __restrict__ out_lp,
                                         int lp_dt, const unsigned char* __restrict__ row_zero, long long rows) {
  pdl_launch_dependents();
  constexpr int C = VEC * 128;
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  // affine parameters are launch constants: fetch them while the producer of the rows is still running
  float4 g[VEC], b[VEC];
  if (gamma != nullptr) {
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      g[i] = __ldg(reinterpret_cast<const float4*>(gamma) + lane + 32 * i);
      b[i] = __ldg(reinterpret_cast<const float4*>(beta) + lane + 32 * i);
    }
  } else {
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      g[i] = make_float4(1.f, 1.f, 1.f, 1.f);
      b[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  pdl_wait();
  if (row >= rows) return;
  const bool zero = row_zero != nullptr && row_zero[row] != 0;
  float4 v[VEC];
  float s = 0.f;
  if (IN_BF16) {
    const uint2* x = reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(in) + row * ld_in);
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const uint2 u = x[lane + 32 * i];
      const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
      const float2 b2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
      v[i] = make_float4(a.x, a.y, b2.x, b2.y);
    }
  } else {
    const float4* x = reinterpret_cast<const float4*>(in + row * ld_in);
#pragma unroll
    for (int i = 0; i < VEC; ++i) v[i] = x[lane + 32 * i];
  }
#pragma unroll
  for (int i = 0; i < VEC; ++i) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  const float mean = warp_sum(s) * (1.f / C);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
    q += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
  }
  const float rstd = rsqrtf(warp_sum(q) * (1.f / C) + eps);
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    const int c4 = lane + 32 * i;
    float4 o;
    o.x = v[i].x * rstd * g[i].x + b[i].x;
    o.y = v[i].y * rstd * g[i].y + b[i].y;
    o.z = v[i].z * rstd * g[i].z + b[i].z;
    o.w = v[i].w * rstd * g[i].w + b[i].w;
    if (zero) o = make_float4(0.f, 0.f, 0.f, 0.f);
    if (out_f32 != nullptr) reinterpret_cast<float4*>(out_f32 + row * C)[c4] = o;
    if (out_lp != nullptr) {
      if (lp_dt == DT_BF16) {
        uint2 u = make_uint2(pack_bf16(o.x, o.y), pack_bf16(o.z, o.w));
        reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(out_lp) + row * C)[c4] = u;
      } else if (lp_dt == DT_F16) {
        __half2 h0 = __floats2half2_rn(o.x, o.y), h1 = __floats2half2_rn(o.z, o.w);
        uint2 u = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
        reinterpret_cast<uint2*>(reinterpret_cast<__half*>(out_lp) + row * C)[c4] = u;
      } else {
        reinterpret_cast<float4*>(reinterpret_cast<float*>(out_lp) + row * C)[c4] = o;
      }
    }
  }
}

// ------------------------------------------------------------------------------------- layout / dtype
__global__ void bct_to_rows_kernel(const void* __restrict__ in, int in_dt, long long sb, long long sc, long long st,
                                   int B, int C, int T, void* __restrict__ out, int out_dt, long long ldo) {
  pdl_launch_dependents();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)B * T * C) return;
  const int c = (int)(i % C);
  const long long bt = i / C;
  const int t = (int)(bt % T);
  const int b = (int)(bt / T);
  store_lp(out, out_dt, bt * ldo + c, load_any(in, in_dt, b * sb + c * sc + t * st));
}

__global__ void convert_kernel(const void* __restrict__ in, int in_dt, void* __restrict__ out, int out_dt,
                               long long n) {
  pdl_launch_dependents();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) store_lp(out, out_dt, i, load_any(in, in_dt, i));
}

// 4 consecutive columns per thread
__global__ void split_rows_kernel(const float* __restrict__ in, long long ld, __nv_bfloat16* __restrict__ out,
                                  int planes, long long rows, int cols, int T, int Tpad) {
  pdl_launch_dependents();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int c4n = cols >> 2;
  if (i >= rows * c4n) return;
  const long long r = i / c4n;
  const int c = (int)(i - r * c4n) * 4;
  const float4 x = *reinterpret_cast<const float4*>(in + r * ld + c);
  const long long orow = T > 0 ? (r / T) * Tpad + (r % T) : r;
  __nv_bfloat16* o = out + orow * ((long long)planes * cols) + c;
  const __nv_bfloat162 h0 = __floats2bfloat162_rn(x.x, x.y), h1 = __floats2bfloat162_rn(x.z, x.w);
  uint2 u = make_uint2(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1));
  *reinterpret_cast<uint2*>(o) = u;
  if (planes > 1) {
    const float2 f0 = __bfloat1622float2(h0), f1 = __bfloat1622float2(h1);
    uint2 m = make_uint2(pack_bf16(x.x - f0.x, x.y - f0.y), pack_bf16(x.z - f1.x, x.w - f1.y));
    *reinterpret_cast<uint2*>(o + cols) = m;
  }
}

// ------------------------------------------------------------------------------------- lip frontend
// Spatial (kh,kw) patches of the Conv3d(1,64,(5,7,7),s(1,2,2),p(2,3,3)) stem (avhubert/resnet.py:138): for
// clip-local frame (bl,t) and output pixel (ho,wo), out row ((bl*(T+2)+t)*1936 + ho*44+wo) holds the 49 taps
// x[t, 2ho+kh-3, 2wo+kw-3] at column kh*7+kw (columns 49..63 zero).  The 5 temporal taps are then row shifts
// of +-1936 rows in the tcgen05 GEMM; the two gap frames after every clip are never written and stay zero.
// One CTA = one frame x 4 output rows (176 pixels): the 13 input rows it needs are staged in smem (zero borders
// included, so the gather has no bounds checks), then every thread assembles 16-byte chunks of 8 taps.
constexpr int SP_ROWS = 4;                 // output rows per CTA
constexpr int SP_IN_ROWS = 2 * SP_ROWS + 5;   // 13 input rows
constexpr int SP_PITCH = 96;               // 88 columns + 3 zero columns left + 5 right
__global__ void __launch_bounds__(256)
stem_patches_kernel(const void* __restrict__ video, int in_dt, int T, int b0, int nb,
                    __nv_bfloat16* __restrict__ out, int planes) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float sIn[SP_IN_ROWS][SP_PITCH];
  const int rg = blockIdx.x % 11;                       // row group: output rows 4*rg .. 4*rg+3
  const long long ft = blockIdx.x / 11;                 // clip-local frame index over the chunk
  const int t = (int)(ft % T);
  const int bl = (int)(ft / T);
  const long long src = ((long long)(b0 + bl) * T + t) * 7744;
  const int h0 = 2 * (rg * SP_ROWS) - 3;                // first input row staged
  for (int i = threadIdx.x; i < SP_IN_ROWS * SP_PITCH; i += 256) {
    const int r = i / SP_PITCH, c = i - r * SP_PITCH;
    const int hh = h0 + r, ww = c - 3;
    float x = 0.f;
    if (hh >= 0 && hh < 88 && ww >= 0 && ww < 88) x = load_any(video, in_dt, src + hh * 88 + ww);
    sIn[r][c] = x;
  }
  __syncthreads();
  const long long orow0 = ((long long)bl * (T + 2) + t) * 1936 + (long long)rg * SP_ROWS * 44;
  for (int i = threadIdx.x; i < SP_ROWS * 44 * 8; i += 256) {
    const int chunk = i & 7;
    const int pl = i >> 3;                              // pixel inside the CTA's 4 rows
    const int hol = pl / 44, wo = pl - hol * 44;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = chunk * 8 + j;
      const int kh = k / 7, kw = k - kh * 7;
      v[j] = k < 49 ? sIn[2 * hol + kh][2 * wo + kw] : 0.f;
    }
    __nv_bfloat162 h[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) h[j] = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
    uint4* o = reinterpret_cast<uint4*>(out + (orow0 + pl) * (64ll * planes));
    o[chunk] = *reinterpret_cast<uint4*>(h);
    if (planes > 1) {
      uint4 m;
      uint32_t* mp = reinterpret_cast<uint32_t*>(&m);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f2 = __bfloat1622float2(h[j]);
        mp[j] = pack_bf16(v[2 * j] - f2.x, v[2 * j + 1] - f2.y);
      }
      o[8 + chunk] = m;
    }
  }
}

__device__ __forceinline__ uint4 bf16x8_max(uint4 a, uint4 b) {
  uint4 r;
  const __nv_bfloat162* pa = reinterpret_cast<const __nv_bfloat162*>(&a);
  const __nv_bfloat162* pb = reinterpret_cast<const __nv_bfloat162*>(&b);
  __nv_bfloat162* pr = reinterpret_cast<__nv_bfloat162*>(&r);
#pragma unroll
  for (int i = 0; i < 4; ++i) pr[i] = __hmax2(pa[i], pb[i]);
  return r;
}
__device__ __forceinline__ float4 f32x4_max(float4 a, float4 b) {
  return make_float4(fmaxf(a.x, b.x), fmaxf(a.y, b.y), fmaxf(a.z, b.z), fmaxf(a.w, b.w));
}

// MaxPool3d((1,3,3),(1,2,2),(0,1,1)) (avhubert/resnet.py:141): [nf,44,44,64] -> padded [nf,23,23,64].
// VT = uint4 (8 bf16) or float4 (4 fp32); CV = vectors per pixel.
template <typename VT, int CV, bool F32>
__global__ void maxpool_stem_kernel(const VT* __restrict__ in, VT* __restrict__ out, int nf, int T) {
  pdl_launch_dependents();
  pdl_wait();
  // one CTA row of threads per frame (blockIdx.y), 32-bit index math inside the frame
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 484u * CV) return;
  const int cv = (int)(i % CV);
  const int pix = (int)(i / CV);
  const long long n = blockIdx.y;
  const int ho = pix / 22, wo = pix - ho * 22;
  const long long ns = (n / T) * (T + 2) + (n % T);      // source frame index in the clip-padded stem output
  VT m;
  bool first = true;
  for (int dh = -1; dh <= 1; ++dh) {
    const int h = 2 * ho + dh;
    if (h < 0 || h >= 44) continue;
    for (int dw = -1; dw <= 1; ++dw) {
      const int w = 2 * wo + dw;
      if (w < 0 || w >= 44) continue;
      const VT v = __ldg(in + ((ns * 44 + h) * 44 + w) * CV + cv);
      if (first) m = v;
      else {
        if constexpr (F32) m = f32x4_max(m, v);
        else m = bf16x8_max(m, v);
      }
      first = false;
    }
  }
  out[((n * 23 + ho) * 23 + wo) * CV + cv] = m;
}

// 3x3 stride-2 pad-1 im2col from the zero-padded layout [n,H+1,W+1,C] (avhubert/resnet.py:15-17 with stride 2)
template <typename IdxT>
__global__ void im2col_s2_kernel(const uint4* __restrict__ in, uint4* __restrict__ out, int n, int H, int W, int C8) {
  pdl_launch_dependents();
  pdl_wait();
  const int Ho = (H + 1) / 2, Wo = (W + 1) / 2;
  const IdxT i = (IdxT)blockIdx.x * blockDim.x + threadIdx.x;
  const IdxT total = (IdxT)n * Ho * Wo * 9 * C8;
  if (i >= total) return;
  // 32-bit index arithmetic whenever the problem allows it: the 64-bit divisions were most of this kernel's time
  const IdxT per_row = (IdxT)(9 * C8);
  const IdxT row = i / per_row;
  const unsigned rem = (unsigned)(i - row * per_row);
  const unsigned tap = rem / (unsigned)C8, c8 = rem - tap * (unsigned)C8;
  const IdxT img = row / (IdxT)(Ho * Wo);
  const unsigned pix = (unsigned)(row - img * (IdxT)(Ho * Wo));
  const int ho = (int)(pix / (unsigned)Wo), wo = (int)(pix - (unsigned)ho * (unsigned)Wo);
  const int h = 2 * ho + (int)(tap / 3) - 1, w = 2 * wo + (int)(tap % 3) - 1;
  uint4 v = make_uint4(0, 0, 0, 0);
  if (h >= 0 && h < H && w >= 0 && w < W)
    v = __ldg(in + (((long long)img * (H + 1) + h) * (W + 1) + w) * C8 + c8);
  out[i] = v;
}

// AdaptiveAvgPool2d(1) (avhubert/resnet.py:90,127) over the valid pixels of a layout with pixel pitch S
__global__ void avgpool_kernel(const void* __restrict__ in, void* __restrict__ out, int dt, int n, int H, int W,
                               int C, int S) {
  pdl_launch_dependents();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)n * C) return;
  const int c = (int)(i % C);
  const long long img = i / C;
  float s = 0.f;
  for (int h = 0; h < H; ++h)
    for (int w = 0; w < W; ++w) s += load_any(in, dt, ((img * S + h) * S + w) * C + c);
  store_lp(out, dt, i, s / (float)(H * W));
}

// Video pre-processing of the dataset's eval transform (avhubert/hubert_dataset.py:222-226,298-302;
// avhubert/utils.py:56-95): uint8 gray frames [n, src_h, src_w] -> x/255 -> centre crop -> (x - mean)/std.  The
// reference does this in float64 numpy and casts to float32 (hubert_dataset.py:432): the 256 possible results are
// computed once per CTA in double and looked up, so fp32 outputs are bit-identical to the reference's.
__global__ void __launch_bounds__(256)
video_preprocess_kernel(const unsigned char* __restrict__ in, void* __restrict__ out, int out_dt, long long n_frames,
                        int src_h, int src_w, int crop, int dh, int dw, double mean, double stdv,
                        const unsigned char* __restrict__ frame_zero) {
  pdl_launch_dependents();
  __shared__ float lut[256];
  lut[threadIdx.x] = (float)((((double)threadIdx.x - 0.0) / 255.0 - mean) / stdv);
  __syncthreads();
  pdl_wait();
  const int groups = crop / 8;                              // 8 output pixels per thread
  const long long total = n_frames * crop * groups;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int g = (int)(i % groups);
  const long long r = i / groups;
  const int y = (int)(r % crop);
  const long long f = r / crop;
  const unsigned char* src = in + (f * src_h + (y + dh)) * (long long)src_w + dw + g * 8;
  float v[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) v[k] = lut[src[k]];
  // the collater zero-pads AFTER the per-sample Normalize (hubert_dataset.py:430-456): pad frames are 0.0 in
  // normalised space, not (0/255 - mean)/std
  if (frame_zero != nullptr && frame_zero[f]) {
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = 0.f;
  }
  const long long o = (f * crop + y) * (long long)crop + g * 8;
  if (out_dt == DT_F32) {
    float4* d = reinterpret_cast<float4*>(reinterpret_cast<float*>(out) + o);
    d[0] = make_float4(v[0], v[1], v[2], v[3]);
    d[1] = make_float4(v[4], v[5], v[6], v[7]);
  } else if (out_dt == DT_BF16) {
    *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(out) + o) =
        make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
  } else {
    __half2 h[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) h[k] = __floats2half2_rn(v[2 * k], v[2 * k + 1]);
    *reinterpret_cast<uint4*>(reinterpret_cast<__half*>(out) + o) = *reinterpret_cast<uint4*>(h);
  }
}

// ------------------------------------------------------------------------------------- packed ragged batches
// Clips sit back to back: cu[b] = first row of clip b, cu[B] = total rows.  (SURVEY 7 step 9: no work on pad frames.)
__device__ __forceinline__ int find_clip(const int* __restrict__ cu, int B, int r) {     // largest b with cu[b] <= r
  int lo = 0, hi = B - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(cu + mid) <= r) lo = mid; else hi = mid - 1;
  }
  return lo;
}
// strided [B, C, Tpitch] -> packed rows [rows_cap, ldo]; rows >= cu[B] are written as zeros
__global__ void bct_to_rows_ragged_kernel(const void* __restrict__ in, int in_dt, long long sb, long long sc, long long st,
                                          int B, int C, const int* __restrict__ cu, void* __restrict__ out, int out_dt,
                                          long long ldo, long long rows_cap) {
  pdl_launch_dependents();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows_cap * C) return;
  const int c = (int)(i % C);
  const int r = (int)(i / C);
  float v = 0.f;
  if (r < __ldg(cu + B)) {
    const int b = find_clip(cu, B, r);
    v = load_any(in, in_dt, b * sb + c * sc + (long long)(r - __ldg(cu + b)) * st);
  }
  store_lp(out, out_dt, (long long)r * ldo + c, v);
}
// residual stream [rows, cols] fp32 -> zero-gapped bf16 layout of the positional conv: clip b occupies padded rows
// [cu[b] + gap*b, +T_b), followed by `gap` zero rows; row_map[padded row] = packed row, or -1 for gap / tail rows
__global__ void pos_pad_ragged_kernel(const float* __restrict__ in, long long ld, __nv_bfloat16* __restrict__ out,
                                      int* __restrict__ row_map, const int* __restrict__ cu, int B, int cols, int gap,
                                      long long rows_pad) {
  pdl_launch_dependents();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int c4n = cols >> 2;
  if (i >= rows_pad * c4n) return;
  const int rp = (int)(i / c4n);
  const int c = (int)(i - (long long)rp * c4n) * 4;
  int lo = 0, hi = B - 1;                       // largest b with cu[b] + gap*b <= rp
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(cu + mid) + gap * mid <= rp) lo = mid; else hi = mid - 1;
  }
  const int t = rp - (__ldg(cu + lo) + gap * lo);
  const int src = (t < __ldg(cu + lo + 1) - __ldg(cu + lo)) ? __ldg(cu + lo) + t : -1;
  uint2 u = make_uint2(0u, 0u);
  if (src >= 0) {
    const float4 x = *reinterpret_cast<const float4*>(in + (long long)src * ld + c);
    u = make_uint2(pack_bf16(x.x, x.y), pack_bf16(x.z, x.w));
  }
  *reinterpret_cast<uint2*>(out + (long long)rp * cols + c) = u;
  if (c == 0) row_map[rp] = src;
}
// packed fp32 rows -> dense [B, T, cols] in out_dt, zeros at the pad positions
__global__ void unpack_rows_kernel(const float* __restrict__ in, const int* __restrict__ cu, void* __restrict__ out, int out_dt,
                                   int B, int T, int cols) {
  pdl_launch_dependents();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int c4n = cols >> 2;
  if (i >= (long long)B * T * c4n) return;
  const long long bt = i / c4n;
  const int c = (int)(i - bt * c4n) * 4;
  const int b = (int)(bt / T), t = (int)(bt - (long long)b * T);
  const int r0 = __ldg(cu + b);
  float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
  if (t < __ldg(cu + b + 1) - r0) x = *reinterpret_cast<const float4*>(in + (long long)(r0 + t) * cols + c);
  const long long o = bt * cols + c;
  if (out_dt == DT_F32) *reinterpret_cast<float4*>(reinterpret_cast<float*>(out) + o) = x;
  else if (out_dt == DT_BF16)
    *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(out) + o) = make_uint2(pack_bf16(x.x, x.y), pack_bf16(x.z, x.w));
  else {
    const __half2 h0 = __floats2half2_rn(x.x, x.y), h1 = __floats2half2_rn(x.z, x.w);
    *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(out) + o) =
        make_uint2(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1));
  }
}

// Per-sample linear resize along time (F.interpolate(mode='linear', align_corners=False) on [1, C, len_in[b]] ->
// len_out[b], src/model.py:601-606) for a whole batch: x [B, T, C] -> out [B, Tout, C], rows >= len_out[b] zero,
// mask[b, t] = t < len_out[b].  Index arithmetic as ATen's upsample_linear1d: scale = in / out (fp32),
// src = max(scale * (t + 0.5) - 0.5, 0), i0 = floor(src), i1 = i0 + (i0 < in - 1), w1 = src - i0.
__global__ void interp_linear_kernel(const void* __restrict__ x, int dt, int B, int T, int C,
                                     const int* __restrict__ len_in, const int* __restrict__ len_out, int Tout,
                                     void* __restrict__ out, long long* __restrict__ mask) {
  pdl_launch_dependents();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)B * Tout * C) return;
  const int c = (int)(i % C);
  const long long bt = i / C;
  const int t = (int)(bt % Tout), b = (int)(bt / Tout);
  const int n_in = len_in[b], n_out = len_out[b];
  float v = 0.f;
  if (t < n_out && n_in > 0) {
    const float scale = (float)n_in / (float)n_out;
    float src = scale * ((float)t + 0.5f) - 0.5f;
    if (src < 0.f) src = 0.f;
    const int i0 = (int)src;
    const int i1 = i0 + (i0 < n_in - 1 ? 1 : 0);
    const float w1 = src - (float)i0, w0 = 1.f - w1;
    const long long base = (long long)b * T * C + c;
    v = w0 * load_any(x, dt, base + (long long)i0 * C) + w1 * load_any(x, dt, base + (long long)i1 * C);
  }
  store_lp(out, dt, i, v);
  if (c == 0 && mask != nullptr) mask[bt] = t < n_out ? 1 : 0;
}

// [rows, cols] of any float dtype -> fp32 residual stream, rows flagged in row_zero written as zeros
__global__ void load_rows_kernel(const void* __restrict__ in, int in_dt, float* __restrict__ out,
                                 const unsigned char* __restrict__ row_zero, long long rows, int cols) {
  pdl_launch_dependents();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * cols) return;
  const long long r = i / cols;
  out[i] = (row_zero != nullptr && row_zero[r]) ? 0.f : load_any(in, in_dt, i);
}

inline int blocks_for(long long n, int per) { return (int)((n + per - 1) / per); }

}  // namespace

int launch_interp_linear(const void* x, int dt, int B, int T, int C, const int* len_in, const int* len_out, int Tout,
                         void* out, long long* mask, cudaStream_t stream) {
  const long long n = (long long)B * Tout * C;
  if (n <= 0) return 0;
  AVH_CUDA_OK(launch_pdl(interp_linear_kernel, dim3(blocks_for(n, 256)), dim3(256), 0, stream, x, dt, B, T, C, len_in, len_out,
                         Tout, out, mask));
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_load_rows(const void* in, int in_dt, float* out, const unsigned char* row_zero, long long rows, int cols,
                     cudaStream_t stream) {
  const long long n = rows * cols;
  if (n <= 0) return 0;
  AVH_CUDA_OK(launch_pdl(load_rows_kernel, dim3(blocks_for(n, 256)), dim3(256), 0, stream, in, in_dt, out, row_zero, rows, cols));
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_bct_to_rows_ragged(const void* in, int in_dt, long long sb, long long sc, long long st, int B, int C,
                              const int* cu, void* out, int out_dt, long long ldo, long long rows_cap, cudaStream_t stream) {
  const long long n = rows_cap * C;
  if (n <= 0) return 0;
  AVH_CUDA_OK(launch_pdl(bct_to_rows_ragged_kernel, dim3(blocks_for(n, 256)), dim3(256), 0, stream, in, in_dt, sb, sc, st, B,
                         C, cu, out, out_dt, ldo, rows_cap));
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_pos_pad_ragged(const float* in, long long ld, void* out, int* row_map, const int* cu, int B, int cols, int gap,
                          long long rows_pad, cudaStream_t stream) {
  AVH_CHECK(cols % 4 == 0 && ld % 4 == 0, "pos_pad needs 4-column granularity");
  const long long n = rows_pad * (cols / 4);
  if (n <= 0) return 0;
  AVH_CUDA_OK(launch_pdl(pos_pad_ragged_kernel, dim3(blocks_for(n, 256)), dim3(256), 0, stream, in, ld,
                         reinterpret_cast<__nv_bfloat16*>(out), row_map, cu, B, cols, gap, rows_pad));
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_unpack_rows(const float* in, const int* cu, void* out, int out_dt, int B, int T, int cols, cudaStream_t stream) {
  AVH_CHECK(cols % 4 == 0, "unpack_rows needs 4-column granularity");
  const long long n = (long long)B * T * (cols / 4);
  if (n <= 0) return 0;
  AVH_CUDA_OK(launch_pdl(unpack_rows_kernel, dim3(blocks_for(n, 256)), dim3(256), 0, stream, in, cu, out, out_dt, B, T, cols));
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_video_preprocess(const unsigned char* frames, long long n_frames, int src_h, int src_w, int crop, double mean,
                            double stdv, void* out, int out_dt, const unsigned char* frame_zero, cudaStream_t stream) {
  if (n_frames <= 0) return 0;
  AVH_CHECK(crop >= 8 && crop % 8 == 0 && crop <= src_h && crop <= src_w, "crop must be a multiple of 8 and fit the frame");
  AVH_CHECK(stdv != 0.0, "std must be non-zero");
  AVH_CHECK((reinterpret_cast<uintptr_t>(out) & 31) == 0, "output must be 32-byte aligned");
  // CenterCrop of the reference: delta = int(round(w - tw) / 2.)  (utils.py:86-88; truncation toward zero)
  const int dh = (src_h - crop) / 2, dw = (src_w - crop) / 2;
  const long long total = n_frames * crop * (crop / 8);
  AVH_CHECK(total / 256 + 1 < (1ll << 31), "too many frames for one launch");
  AVH_CUDA_OK(launch_pdl(video_preprocess_kernel, dim3((unsigned)blocks_for(total, 256)), dim3(256), 0, stream, frames, out,
                         out_dt, n_frames, src_h, src_w, crop, dh, dw, mean, stdv, frame_zero));
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_layernorm(const void* in, int in_dt, long long ld_in, const float* gamma, const float* beta, float eps,
                     float* out_f32, void* out_lp, int lp_dt, const unsigned char* row_zero, long long rows, int C,
                     cudaStream_t stream) {
  const int wpb = 4;
  if (rows <= 0) return 0;
  const int grid = blocks_for(rows, wpb);
  const bool vec_ok = in_dt == DT_F32 && C % 128 == 0 && ld_in % 4 == 0 &&
                      (reinterpret_cast<uintptr_t>(in) & 15) == 0;
#define AVH_LN_VEC(V)                                                                                            \
  AVH_CUDA_OK(launch_pdl(layernorm_f32_vec_kernel<V>, dim3(grid), dim3(wpb * 32), 0, stream,                    \
                         reinterpret_cast<const float*>(in), ld_in, gamma, beta, eps, out_f32, out_lp, lp_dt, row_zero, rows))
  if (vec_ok && C == 768) AVH_LN_VEC(6);
  else if (vec_ok && C == 1024) AVH_LN_VEC(8);
  else if (vec_ok && C == 1536) AVH_LN_VEC(12);
  else if (vec_ok && C == 2048) AVH_LN_VEC(16);
  else if (vec_ok && C == 256) AVH_LN_VEC(2);
  else if (vec_ok && C == 128) AVH_LN_VEC(1);
  else if (in_dt == DT_BF16 && ld_in % 4 == 0 && (reinterpret_cast<uintptr_t>(in) & 7) == 0 && (C == 2048 || C == 1536 || C == 1024 || C == 768)) {
#define AVH_LN_VECB(V)                                                                                           \
  AVH_CUDA_OK(launch_pdl(layernorm_f32_vec_kernel<V, true>, dim3(grid), dim3(wpb * 32), 0, stream,                \
                         reinterpret_cast<const float*>(in), ld_in, gamma, beta, eps, out_f32, out_lp, lp_dt, row_zero, rows))
    if (C == 2048) AVH_LN_VECB(16);
    else if (C == 1536) AVH_LN_VECB(12);
    else if (C == 1024) AVH_LN_VECB(8);
    else AVH_LN_VECB(6);
#undef AVH_LN_VECB
  } else
    AVH_CUDA_OK(launch_pdl(layernorm_kernel, dim3(grid), dim3(wpb * 32), 0, stream, in, in_dt, ld_in, gamma, beta, eps,
                           out_f32, out_lp, lp_dt, row_zero, rows, C));
#undef AVH_LN_VEC
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_bct_to_rows(const void* in, int in_dt, long long sb, long long sc, long long st, int B, int C, int T,
                       void* out, int out_dt, long long ldo, cudaStream_t stream) {
  const long long n = (long long)B * C * T;
  if (n <= 0) return 0;
  AVH_CUDA_OK(launch_pdl(bct_to_rows_kernel, dim3(blocks_for(n, 256)), dim3(256), 0, stream, in, in_dt, sb, sc, st, B, C,
                         T, out, out_dt, ldo));
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_convert(const void* in, int in_dt, void* out, int out_dt, long long n, cudaStream_t stream) {
  if (n <= 0) return 0;
  AVH_CUDA_OK(launch_pdl(convert_kernel, dim3(blocks_for(n, 256)), dim3(256), 0, stream, in, in_dt, out, out_dt, n));
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_split_rows(const float* in, long long ld, void* out, int planes, long long rows, int cols, int T,
                      int Tpad, cudaStream_t stream) {
  AVH_CHECK(cols % 4 == 0 && ld % 4 == 0, "split_rows needs 4-column granularity");
  const long long n = rows * (cols / 4);
  if (n <= 0) return 0;
  AVH_CUDA_OK(launch_pdl(split_rows_kernel, dim3(blocks_for(n, 256)), dim3(256), 0, stream, in, ld,
                         reinterpret_cast<__nv_bfloat16*>(out), planes, rows, cols, T, Tpad));
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_stem_patches(const void* video, int in_dt, int T, int b0, int nb, void* out, int planes,
                        cudaStream_t stream) {
  const long long nblk = (long long)nb * T * 11;
  if (nblk <= 0) return 0;
  AVH_CUDA_OK(launch_pdl(stem_patches_kernel, dim3((unsigned)nblk), dim3(256), 0, stream, video, in_dt, T, b0, nb,
                         reinterpret_cast<__nv_bfloat16*>(out), planes));
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_maxpool_stem(const void* in, void* out, int nf, int T, int fp32, cudaStream_t stream) {
  if (nf <= 0) return 0;
  if (fp32) {
    AVH_CUDA_OK(launch_pdl(maxpool_stem_kernel<float4, 16, true>, dim3(blocks_for(484 * 16, 256), nf), dim3(256), 0, stream,
                           reinterpret_cast<const float4*>(in), reinterpret_cast<float4*>(out), nf, T));
  } else {
    AVH_CUDA_OK(launch_pdl(maxpool_stem_kernel<uint4, 8, false>, dim3(blocks_for(484 * 8, 256), nf), dim3(256), 0, stream,
                           reinterpret_cast<const uint4*>(in), reinterpret_cast<uint4*>(out), nf, T));
  }
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_im2col_s2(const void* in, void* out, int n, int H, int W, int C, cudaStream_t stream) {
  const int Ho = (H + 1) / 2, Wo = (W + 1) / 2;
  const long long total = (long long)n * Ho * Wo * 9 * (C / 8);
  if (total <= 0) return 0;
  if (total < (1ll << 31))
    AVH_CUDA_OK(launch_pdl(im2col_s2_kernel<unsigned>, dim3(blocks_for(total, 256)), dim3(256), 0, stream,
                           reinterpret_cast<const uint4*>(in), reinterpret_cast<uint4*>(out), n, H, W, C / 8));
  else
    AVH_CUDA_OK(launch_pdl(im2col_s2_kernel<long long>, dim3(blocks_for(total, 256)), dim3(256), 0, stream,
                           reinterpret_cast<const uint4*>(in), reinterpret_cast<uint4*>(out), n, H, W, C / 8));
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

int launch_avgpool(const void* in, void* out, int n, int H, int W, int C, int pitch, int fp32, cudaStream_t stream) {
  const long long total = (long long)n * C;
  if (total <= 0) return 0;
  AVH_CUDA_OK(launch_pdl(avgpool_kernel, dim3(blocks_for(total, 256)), dim3(256), 0, stream, in, out,
                         fp32 ? DT_F32 : DT_BF16, n, H, W, C, pitch));
  AVH_CUDA_OK(cudaGetLastError());
  count_launch(1);
  return 0;
}

}  // namespace avh
