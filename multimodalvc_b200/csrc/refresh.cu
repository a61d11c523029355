// Weight refresh on the device for trainable handles: after an optimizer step the parameters live in the caller's
// device tensors; these kernels rewrite the PACKED copies the training plans read (K-major bf16 planes of every Linear /
// convolution and their transposes, fp32 vectors, the weight-normed positional convolution) IN PLACE, so that plans and
// captured graphs stay valid and no byte crosses the host.  Layouts are the ones pack_all (api.cu) produces on the host:
// each kernel is the index map of one packer.  (avh_finalize_weights re-packs everything through the host: 6 s for the
// Large model against a 32 ms training step.)  Before the first eval forward after training, the eval-only forms
// (BatchNorm folds, the conv2 + shortcut GEMM weights) are recomputed here too, bit-identical to the host packers.
#include "common.cuh"
#include "kernels.h"

#include <cuda_fp16.h>

namespace avh {
namespace {

__device__ __forceinline__ float ldw(const void* p, int dt, long long i) {
  if (dt == DT_BF16) return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[i]);
  if (dt == DT_F16) return __half2float(reinterpret_cast<const __half*>(p)[i]);
  return reinterpret_cast<const float*>(p)[i];
}
// plane 0 = bf16 round, plane 1 (planes == 2) = bf16 of the remainder, `ps` elements further
__device__ __forceinline__ void st_planes(__nv_bfloat16* out, long long i, long long ps, int planes, float v) {
  const __nv_bfloat16 hi = __float2bfloat16_rn(v);
  out[i] = hi;
  if (planes > 1) out[i + ps] = __float2bfloat16_rn(v - __bfloat162float(hi));
}

// src [n, k] -> dst rows row0 .. row0+n of [*, planes*ld] (transposed: dst[c, col0 + r] of [k, planes*ld])
__global__ void __launch_bounds__(256)
refresh_matrix_kernel(const void* __restrict__ src, int dt, long long n, long long k, float scale, __nv_bfloat16* __restrict__ dst,
                      long long ld, int planes, long long off, int transposed) {
  const long long total = n * k;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const long long r = i / k, c = i % k;
    const float v = ldw(src, dt, i) * scale;
    const long long d = transposed ? c * planes * ld + off + r : (off + r) * planes * ld + c;
    st_planes(dst, d, ld, planes, v);
  }
}
// src [n_src] (n_src == 1: broadcast) -> dst float [n]
__global__ void refresh_vec_kernel(const void* __restrict__ src, int dt, long long n, long long n_src, float scale,
                                   float* __restrict__ dst) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = ldw(src, dt, n_src == 1 ? 0 : i) * scale;
}
// conv weight [cout, cin, ks, ks] -> [cout, planes*K] with K index (tap, cin); transposed: [K, planes*ld] with column cout
__global__ void __launch_bounds__(256)
refresh_conv_kernel(const void* __restrict__ src, int dt, int cout, int cin, int ksq, __nv_bfloat16* __restrict__ dst, long long ld,
                    int planes, int transposed) {
  const long long total = (long long)cout * cin * ksq;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int t = (int)(i % ksq);
    const long long oc = i / ksq;
    const int c = (int)(oc % cin), o = (int)(oc / cin);
    const long long kidx = (long long)t * cin + c;
    const long long d = transposed ? kidx * planes * ld + o : (long long)o * planes * ld + kidx;
    st_planes(dst, d, ld, planes, ldw(src, dt, i));
  }
}
// stem Conv3d weight [64, 1, 5, 7, 7] -> [64, planes*320], column dt*64 + kh*7 + kw (pitch8 = 0: the row-shift GEMM
// form) or dt*64 + kh*8 + kw (pitch8 = 1: the fused inference stem and the training patches)
__global__ void refresh_stem_kernel(const void* __restrict__ src, int dt, __nv_bfloat16* __restrict__ dst, int planes, int pitch8) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 64 * 245) return;
  const int o = i / 245, rem = i % 245, d = rem / 49, j = rem % 49;
  const int col = pitch8 ? (j / 7) * 8 + j % 7 : j;
  st_planes(dst, (long long)o * planes * 320 + d * 64 + col, 320, planes, ldw(src, dt, i));
}
// weight_norm(dim=2): ratio[k] = g[k] / || v[:, :, k] ||   (one CTA per tap, fixed summation order)
__global__ void __launch_bounds__(256)
posconv_ratio_kernel(const void* __restrict__ v, int v_dt, const void* __restrict__ g, int g_dt, long long per_tap, int KT,
                     float* __restrict__ ratio) {
  __shared__ double part[256];
  const int k = blockIdx.x;
  double s = 0.0;
  for (long long i = threadIdx.x; i < per_tap; i += 256) {
    const double x = (double)ldw(v, v_dt, i * KT + k);
    s += x * x;
  }
  part[threadIdx.x] = s;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (threadIdx.x < w) part[threadIdx.x] += part[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) ratio[k] = (float)((double)ldw(g, g_dt, k) / sqrt(part[0]));
}
// grouped positional conv weight_v [D, cg, KT] * ratio -> per-N-tile windowed K-major [D, planes * KT * window]:
// forward: row o, column k*window + (g*cg + i - acol[o/64]);  transposed (dgrad): row g*cg + i, column k*window + (o - acol[row/64])
__global__ void __launch_bounds__(256)
refresh_pos_kernel(const void* __restrict__ v, int dt, const float* __restrict__ ratio, const int* __restrict__ acol, int D, int cg,
                   int KT, int window, __nv_bfloat16* __restrict__ dst, int planes, int transposed) {
  const long long total = (long long)D * cg * KT;
  const long long ld = (long long)KT * window;
  for (long long idx = (long long)blockIdx.x * 256 + threadIdx.x; idx < total; idx += (long long)gridDim.x * 256) {
    const int k = (int)(idx % KT);
    const long long oi = idx / KT;
    const int i = (int)(oi % cg), o = (int)(oi / cg), g = o / cg;
    const float val = ldw(v, dt, idx) * ratio[k];
    long long row, col;
    if (!transposed) { row = o; col = (long long)k * window + (g * cg + i - acol[o / 64]); }
    else { const int ig = g * cg + i; row = ig; col = (long long)k * window + (o - acol[ig / 64]); }
    st_planes(dst, row * planes * ld + col, ld, planes, val);
  }
}

// Eval-mode BatchNorm fold per channel, exactly as the host packers compute it (pack_conv, the stem, bn_fold in
// pack_all): inv = 1 / sqrt(var + 1e-5f), scale = gamma * inv, bias = beta - mean * scale, every operation rounded on
// its own (the intrinsics keep nvcc from contracting into an FMA, which the host code does not do either).  Also
// writes the fp32 copies the training-mode BatchNorm starts from.
__global__ void bn_fold_kernel(const void* __restrict__ g, int g_dt, const void* __restrict__ b, int b_dt,
                               const void* __restrict__ m, int m_dt, const void* __restrict__ v, int v_dt, int C,
                               float* __restrict__ scale, float* __restrict__ bias, float* __restrict__ gamma,
                               float* __restrict__ beta, float* __restrict__ rmean, float* __restrict__ rvar) {
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= C) return;
  const float gv = ldw(g, g_dt, o), bv = ldw(b, b_dt, o), mv = ldw(m, m_dt, o), vv = ldw(v, v_dt, o);
  const float inv = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(vv, 1e-5f)));
  const float sc = __fmul_rn(gv, inv);
  scale[o] = sc;
  bias[o] = __fsub_rn(bv, __fmul_rn(mv, sc));
  gamma[o] = gv; beta[o] = bv; rmean[o] = mv; rvar[o] = vv;
}
// conv2 + 1x1 shortcut as one GEMM (bf16 frame-row path): [cout, planes*K], K = 9*cmid + cin; column t*cmid + c holds
// s2[o] * w2[o, c, t], column 9*cmid + c holds sd[o] * wd[o, c]; bias[o] = b2[o] + bd[o] (the folds of bn_fold_kernel)
__global__ void __launch_bounds__(256)
refresh_c2ds_kernel(const void* __restrict__ w2, int w2_dt, const void* __restrict__ wd, int wd_dt, const float* __restrict__ s2,
                    const float* __restrict__ b2, const float* __restrict__ sd, const float* __restrict__ bd, int cout, int cmid,
                    int cin, __nv_bfloat16* __restrict__ dst, int planes, float* __restrict__ bias) {
  const long long K = 9LL * cmid + cin;
  const long long total = (long long)cout * K;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int o = (int)(i / K);
    const long long kidx = i % K;
    float val;
    if (kidx < 9LL * cmid) {
      const int t = (int)(kidx / cmid), c = (int)(kidx % cmid);
      val = __fmul_rn(s2[o], ldw(w2, w2_dt, ((long long)o * cmid + c) * 9 + t));
    } else {
      val = __fmul_rn(sd[o], ldw(wd, wd_dt, (long long)o * cin + (kidx - 9LL * cmid)));
    }
    st_planes(dst, (long long)o * planes * K + kidx, K, planes, val);
    if (kidx == 0) bias[o] = __fadd_rn(b2[o], bd[o]);
  }
}

inline unsigned grid_of(long long n) {
  const long long b = (n + 255) / 256;
  return (unsigned)(b < 148 * 16 ? (b > 0 ? b : 1) : 148 * 16);
}

}  // namespace

int launch_refresh_matrix(const void* src, int dt, long long n, long long k, float scale, void* dst, long long ld, int planes,
                          long long off, int transposed, cudaStream_t stream) {
  if (n * k <= 0) return 0;
  if (transposed && planes == 1 && (dt == DT_BF16 || dt == DT_F32) && n % 64 == 0 && k % 8 == 0 && ld % 8 == 0 && off % 8 == 0 &&
      (reinterpret_cast<uintptr_t>(src) & 15) == 0)      // 64 x 64 smem tiles, 16-byte accesses on both sides
    return launch_transposeT(src, dt, k, n, (int)k, reinterpret_cast<__nv_bfloat16*>(dst) + off, n, ld, stream, scale);
  refresh_matrix_kernel<<<grid_of(n * k), 256, 0, stream>>>(src, dt, n, k, scale, reinterpret_cast<__nv_bfloat16*>(dst), ld, planes,
                                                            off, transposed);
  AVH_CUDA_OK(cudaGetLastError());
  return 0;
}
int launch_refresh_vec(const void* src, int dt, long long n, long long n_src, float scale, float* dst, cudaStream_t stream) {
  if (n <= 0) return 0;
  refresh_vec_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(src, dt, n, n_src, scale, dst);
  AVH_CUDA_OK(cudaGetLastError());
  return 0;
}
int launch_refresh_conv(const void* src, int dt, int cout, int cin, int ksq, void* dst, long long ld, int planes, int transposed,
                        cudaStream_t stream) {
  refresh_conv_kernel<<<grid_of((long long)cout * cin * ksq), 256, 0, stream>>>(src, dt, cout, cin, ksq,
                                                                               reinterpret_cast<__nv_bfloat16*>(dst), ld, planes,
                                                                               transposed);
  AVH_CUDA_OK(cudaGetLastError());
  return 0;
}
int launch_refresh_stem(const void* src, int dt, void* dst, int planes, int pitch8, cudaStream_t stream) {
  refresh_stem_kernel<<<(64 * 245 + 255) / 256, 256, 0, stream>>>(src, dt, reinterpret_cast<__nv_bfloat16*>(dst), planes, pitch8);
  AVH_CUDA_OK(cudaGetLastError());
  return 0;
}
int launch_posconv_ratio(const void* v, int v_dt, const void* g, int g_dt, long long per_tap, int KT, float* ratio,
                         cudaStream_t stream) {
  posconv_ratio_kernel<<<KT, 256, 0, stream>>>(v, v_dt, g, g_dt, per_tap, KT, ratio);
  AVH_CUDA_OK(cudaGetLastError());
  return 0;
}
int launch_refresh_pos(const void* v, int dt, const float* ratio, const int* acol, int D, int cg, int KT, int window, void* dst,
                       int planes, int transposed, cudaStream_t stream) {
  refresh_pos_kernel<<<grid_of((long long)D * cg * KT), 256, 0, stream>>>(v, dt, ratio, acol, D, cg, KT, window,
                                                                         reinterpret_cast<__nv_bfloat16*>(dst), planes, transposed);
  AVH_CUDA_OK(cudaGetLastError());
  return 0;
}
int launch_bn_fold(const void* g, int g_dt, const void* b, int b_dt, const void* m, int m_dt, const void* v, int v_dt, int C,
                   float* scale, float* bias, float* gamma, float* beta, float* rmean, float* rvar, cudaStream_t stream) {
  if (C <= 0) return 0;
  bn_fold_kernel<<<(C + 255) / 256, 256, 0, stream>>>(g, g_dt, b, b_dt, m, m_dt, v, v_dt, C, scale, bias, gamma, beta, rmean, rvar);
  AVH_CUDA_OK(cudaGetLastError());
  return 0;
}
int launch_refresh_c2ds(const void* w2, int w2_dt, const void* wd, int wd_dt, const float* s2, const float* b2, const float* sd,
                        const float* bd, int cout, int cmid, int cin, void* dst, int planes, float* bias, cudaStream_t stream) {
  refresh_c2ds_kernel<<<grid_of((long long)cout * (9LL * cmid + cin)), 256, 0, stream>>>(
      w2, w2_dt, wd, wd_dt, s2, b2, sd, bd, cout, cmid, cin, reinterpret_cast<__nv_bfloat16*>(dst), planes, bias);
  AVH_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace avh
