// Dropout of the training step (avh_encoder_train_forward / avh_tail_train_forward / avh_full_train_forward and their
// backward): the masks of the no-grad training forward (philox.cuh), applied where the step's forward produces the
// value and regenerated, never stored, where its backward needs them.  The seed is read from a plan-owned device word,
// so a launch list captured into a CUDA graph for one call replays for the seed of any later call.
//
//   masked_gelu      out = m * ((res ? res : 0) + GELU(u))     positional-conv block (x1), activation dropout (g)
//   dropout_residual y = (r ? r : 0) + m * a                   dropout1 / dropout3 before the residual add, dropout_input
//   masked_gelu_bwd  du = m * dg * GELU'(u)                    backward of the activation dropout + GELU
//   dropout_grad     out = m * dx, and its GEMM operand planes backward of a dropout on a block output
//
// Thread = 4 consecutive elements = one Philox call (n and the row width are multiples of 4).
#include "common.cuh"
#include "kernels.h"
#include "philox.cuh"

namespace avh {
namespace {

__device__ __forceinline__ float ld_val(const void* p, int dt, long long i) {
  return dt == DT_BF16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[i]) : reinterpret_cast<const float*>(p)[i];
}
__device__ __forceinline__ void st_val(void* p, int dt, long long i, float v) {
  if (dt == DT_BF16) reinterpret_cast<__nv_bfloat16*>(p)[i] = __float2bfloat16_rn(v);
  else reinterpret_cast<float*>(p)[i] = v;
}
__device__ __forceinline__ float gelu_exact(float u) { return 0.5f * u * (1.f + erff(u * 0.70710678118654752f)); }
__device__ __forceinline__ float gelu_deriv(float u) {
  const float cdf = 0.5f * (1.f + erff(u * 0.70710678118654752f));
  const float pdf = 0.3989422804014327f * __expf(-0.5f * u * u);
  return cdf + u * pdf;
}
__device__ __forceinline__ float lane(const float4& v, int k) { return k == 0 ? v.x : (k == 1 ? v.y : (k == 2 ? v.z : v.w)); }

__global__ void __launch_bounds__(256)
masked_gelu_kernel(const void* __restrict__ u, int u_dt, const float* __restrict__ res, void* __restrict__ out, int out_dt,
                   long long n4, float p, const unsigned long long* __restrict__ seed, unsigned int site) {
  pdl_launch_dependents();
  pdl_wait();
  const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n4) return;
  const float4 m = dropout_mask4(*seed, b, site, p);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const long long i = b * 4 + k;
    st_val(out, out_dt, i, lane(m, k) * ((res ? res[i] : 0.f) + gelu_exact(ld_val(u, u_dt, i))));
  }
}

__global__ void __launch_bounds__(256)
dropout_residual_kernel(const float* __restrict__ r, const float* a, float* y, long long n4, float p,
                        const unsigned long long* __restrict__ seed, unsigned int site) {
  pdl_launch_dependents();
  pdl_wait();
  const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n4) return;
  const float4 m = dropout_mask4(*seed, b, site, p);
  const float4 av = reinterpret_cast<const float4*>(a)[b];
  const float4 rv = r ? reinterpret_cast<const float4*>(r)[b] : make_float4(0.f, 0.f, 0.f, 0.f);
  reinterpret_cast<float4*>(y)[b] = make_float4(rv.x + m.x * av.x, rv.y + m.y * av.y, rv.z + m.z * av.z, rv.w + m.w * av.w);
}

__global__ void __launch_bounds__(256)
masked_gelu_bwd_kernel(const void* __restrict__ u, int u_dt, const void* __restrict__ dg, int dg_dt, void* __restrict__ du,
                       int du_dt, long long n4, float p, const unsigned long long* __restrict__ seed, unsigned int site) {
  pdl_launch_dependents();
  pdl_wait();
  const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n4) return;
  const float4 m = dropout_mask4(*seed, b, site, p);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const long long i = b * 4 + k;
    st_val(du, du_dt, i, lane(m, k) * ld_val(dg, dg_dt, i) * gelu_deriv(ld_val(u, u_dt, i)));
  }
}

// out = m * dx (fp32, may alias dx); op (optional): the bf16 operand planes of out, [rows, planes * C] as split_rows
// writes them (plane 0 = bf16(v), plane 1 = bf16(v - plane 0))
__global__ void __launch_bounds__(256)
dropout_grad_kernel(const float* dx, float* out, __nv_bfloat16* __restrict__ op, int planes, int C, long long n4, float p,
                    const unsigned long long* __restrict__ seed, unsigned int site) {
  pdl_launch_dependents();
  pdl_wait();
  const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n4) return;
  const float4 m = dropout_mask4(*seed, b, site, p);
  const float4 g = reinterpret_cast<const float4*>(dx)[b];
  const float4 v = make_float4(m.x * g.x, m.y * g.y, m.z * g.z, m.w * g.w);
  reinterpret_cast<float4*>(out)[b] = v;
  if (op == nullptr) return;
  const long long i = b * 4;
  const long long r = i / C;
  const int c = (int)(i - r * C);
  __nv_bfloat16* o = op + r * ((long long)planes * C) + c;
  const __nv_bfloat162 h0 = __floats2bfloat162_rn(v.x, v.y), h1 = __floats2bfloat162_rn(v.z, v.w);
  *reinterpret_cast<uint2*>(o) = make_uint2(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1));
  if (planes > 1) {
    const float2 f0 = __bfloat1622float2(h0), f1 = __bfloat1622float2(h1);
    *reinterpret_cast<uint2*>(o + C) = make_uint2(pack_bf16(v.x - f0.x, v.y - f0.y), pack_bf16(v.z - f1.x, v.w - f1.y));
  }
}

inline unsigned grid_for(long long n4) { return (unsigned)((n4 + 255) / 256); }

int check_args(long long n, float p, const unsigned long long* seed) {
  AVH_CHECK(p > 0.f && p < 1.f, "dropout probability must be in (0, 1) (p = 0 launches nothing)");
  AVH_CHECK(n % 4 == 0, "dropout tensors hold a multiple of 4 elements");
  AVH_CHECK(seed != nullptr, "null seed word");
  return 0;
}

}  // namespace

int launch_masked_gelu(const void* u, int u_dt, const float* res, void* out, int out_dt, long long n, float p,
                       const unsigned long long* seed, unsigned int site, cudaStream_t stream) {
  if (check_args(n, p, seed)) return 1;
  AVH_CHECK((u_dt == DT_F32 || u_dt == DT_BF16) && (out_dt == DT_F32 || out_dt == DT_BF16), "masked_gelu: fp32 / bf16 only");
  if (n <= 0) return 0;
  AVH_CUDA_OK(launch_pdl(masked_gelu_kernel, dim3(grid_for(n / 4)), dim3(256), 0, stream, u, u_dt, res, out, out_dt, n / 4, p,
                         seed, site));
  count_launch(1);
  return 0;
}

int launch_dropout_residual(const float* r, const float* a, float* y, long long n, float p, const unsigned long long* seed,
                            unsigned int site, cudaStream_t stream) {
  if (check_args(n, p, seed)) return 1;
  if (n <= 0) return 0;
  AVH_CUDA_OK(launch_pdl(dropout_residual_kernel, dim3(grid_for(n / 4)), dim3(256), 0, stream, r, a, y, n / 4, p, seed, site));
  count_launch(1);
  return 0;
}

int launch_masked_gelu_bwd(const void* u, int u_dt, const void* dg, int dg_dt, void* du, int du_dt, long long n, float p,
                           const unsigned long long* seed, unsigned int site, cudaStream_t stream) {
  if (check_args(n, p, seed)) return 1;
  AVH_CHECK((u_dt == DT_F32 || u_dt == DT_BF16) && (dg_dt == DT_F32 || dg_dt == DT_BF16) && (du_dt == DT_F32 || du_dt == DT_BF16),
            "masked_gelu_bwd: fp32 / bf16 only");
  if (n <= 0) return 0;
  AVH_CUDA_OK(launch_pdl(masked_gelu_bwd_kernel, dim3(grid_for(n / 4)), dim3(256), 0, stream, u, u_dt, dg, dg_dt, du, du_dt,
                         n / 4, p, seed, site));
  count_launch(1);
  return 0;
}

int launch_dropout_grad(const float* dx, float* out, void* op, int planes, long long rows, int C, float p,
                        const unsigned long long* seed, unsigned int site, cudaStream_t stream) {
  const long long n = rows * C;
  if (check_args(n, p, seed)) return 1;
  AVH_CHECK(C % 4 == 0, "dropout_grad: row width must be a multiple of 4");
  if (n <= 0) return 0;
  AVH_CUDA_OK(launch_pdl(dropout_grad_kernel, dim3(grid_for(n / 4)), dim3(256), 0, stream, dx, out,
                         reinterpret_cast<__nv_bfloat16*>(op), planes, C, n / 4, p, seed, site));
  count_launch(1);
  return 0;
}

}  // namespace avh
