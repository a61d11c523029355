// Micro-test of the block-scaled FP8 MMA (tcgen05.mma .kind::mxf8f6f4.block_scale, E4M3 x E4M3, UE8M0 scales per 32 K):
// (1) one 128 x N x 128 product against a host reference with scales that differ per row and per 32-K sub-block, which
//     checks where the scale factors sit in tensor memory, and (2) the issue rate against kind::f16.
//   nvcc -std=c++17 -gencode arch=compute_100a,code=sm_100a -O2 -o mma_mxf8 mma_mxf8.cu && ./mma_mxf8
// Scale layout (row r, 32-K sub-block j of the 128-K block): a 512-byte smem atom per 128 rows
// ((r % 32) * 16 + (r / 32) * 4 + j) moved with tcgen05.cp .32x128b.warpx4, i.e. lane r % 32 of every lane quarter,
// column r / 32, byte j; B rows 128..255 in a second atom 4 columns further.  The MMA of sub-block j selects byte j
// through the scale-factor ids of the instruction descriptor (A: bits 29-30, B: bits 4-5).
#include <cstdio>
#include <cstdint>
#include <vector>
#include <cuda_runtime.h>
#include <cuda_fp8.h>
#include "../../multimodalvc_b200/csrc/common.cuh"
namespace avh { void set_last_error(const std::string&) {} int device_sm_count() { return 148; } void count_launch(int) {} }
using namespace avh;

// Instruction descriptor of kind::mxf8f6f4: E4M3 x E4M3 -> fp32 (formats 0), both K-major, UE8M0 scales (bit 23);
// sf = byte of the scale-factor columns that holds this instruction's 32-K sub-block, for A and for B
__host__ __device__ constexpr uint32_t umma_idesc_mxf8(int M, int N, int sf) {
  return ((uint32_t)sf << 4) | ((uint32_t)(N >> 3) << 17) | (1u << 23) | ((uint32_t)(M >> 4) << 24) | ((uint32_t)sf << 29);
}
__device__ __forceinline__ void umma_mxf8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t tmem_sfa,
                                          uint32_t tmem_sfb, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::mxf8f6f4.block_scale [%0], %1, %2, %3, [%4], [%5], p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(tmem_sfa), "r"(tmem_sfb), "r"(accumulate)
      : "memory");
}
// source descriptor of one 512-byte scale atom: 32 rows x 16 bytes, rows 16 B apart, no swizzle
__device__ __forceinline__ uint64_t umma_desc_sf(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;                   // leading byte offset: 16 B (one column of core matrices)
  d |= (uint64_t)(128 >> 4) << 32;          // stride byte offset: 8 rows x 16 B
  d |= (uint64_t)1 << 46;
  return d;
}
// smem atom -> 32 lanes x 4 columns of tensor memory, replicated into the 4 lane quarters
__device__ __forceinline__ void tmem_cp_sf(uint32_t taddr, uint64_t sdesc) {
  asm volatile("tcgen05.cp.cta_group::1.32x128b.warpx4 [%0], %1;" ::"r"(taddr), "l"(sdesc) : "memory");
}

__host__ __device__ inline int aval(int m, int k) { return (m * 3 + k * 5) % 7 - 3; }
__host__ __device__ inline int bval(int n, int k) { return (n + 2 * k) % 5 - 2; }
__host__ __device__ inline int aexp(int m, int j) { return (m * 7 + j * 3) % 5 - 2; }
__host__ __device__ inline int bexp(int n, int j) { return (n * 3 + j) % 4 - 1; }

// D[128 x N] = sum_k A[m,k] 2^aexp(m,k/32) * B[n,k] 2^bexp(n,k/32), K = 128
__global__ void __launch_bounds__(128, 1) mx_check(int N, float* out) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  uint8_t* sa = smem;                 // 16 KB
  uint8_t* sb = smem + 16384;         // N x 128 B
  uint8_t* ssf = sb + 256 * 128;      // SFA atom (512 B) + SFB atoms
  __shared__ uint64_t bar;
  __shared__ uint32_t slot;
  const int warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < (128 + N) * 8; i += 128) {
    const bool isa = i < 128 * 8;
    const int r = (isa ? i : i - 128 * 8) >> 3, c = i & 7;
    uint8_t v[16];
    for (int e = 0; e < 16; ++e) {
      const int k = c * 16 + e;
      v[e] = __nv_fp8_e4m3((float)(isa ? aval(r, k) : bval(r, k))).__x;
    }
    *reinterpret_cast<uint4*>((isa ? sa : sb) + r * 128 + ((c ^ (r & 7)) << 4)) = *reinterpret_cast<uint4*>(v);
  }
  for (int i = threadIdx.x; i < 128 + N; i += 128) {
    const bool isa = i < 128;
    const int r = isa ? i : i - 128;
    uint8_t* atom = ssf + (isa ? 0 : 512 * (1 + r / 128));
    for (int j = 0; j < 4; ++j)
      atom[(r & 31) * 16 + ((r >> 5) & 3) * 4 + j] = (uint8_t)(127 + (isa ? aexp(r, j) : bexp(r, j)));
  }
  fence_proxy_async_smem();
  if (threadIdx.x == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
  if (warp == 0) tmem_alloc(&slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = slot;
  const uint32_t tsfa = tmem + 256, tsfb = tmem + 264;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 0) {
    if (elect_one()) {
      tmem_cp_sf(tsfa, umma_desc_sf(smem_u32(ssf)));
      for (int b = 0; b < N / 128; ++b) tmem_cp_sf(tsfb + 4 * b, umma_desc_sf(smem_u32(ssf + 512 * (1 + b))));
      const uint64_t ad = umma_desc_sw128(smem_u32(sa)), bd = umma_desc_sw128(smem_u32(sb));
      for (int k = 0; k < 4; ++k) {
        umma_mxf8(tmem, ad + 2 * k, bd + 2 * k, umma_idesc_mxf8(128, N, k), tsfa, tsfb, k != 0);
      }
      umma_commit(&bar);
    }
    __syncwarp();
  }
  mbar_wait(&bar, 0);
  tc_fence_after();
  for (int c0 = 0; c0 < N; c0 += 32) {
    uint32_t v[32];
    tmem_ld_32x32(tmem + ((uint32_t)(warp * 32) << 16) + c0, v);
    tmem_ld_wait();
    for (int j = 0; j < 32; ++j) out[(size_t)threadIdx.x * 256 + c0 + j] = __uint_as_float(v[j]);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512);
}

// clk per MMA over a 128-K (fp8) / 64-K (bf16) k-block of 4 instructions; kind 0 = f16, 1 = mxf8f6f4.block_scale
__global__ void __launch_bounds__(128, 1) rate(int N, int kind, int iters, long long* out) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  __shared__ uint64_t bar;
  __shared__ uint32_t slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < 64 * 1024 / 4; i += 128) reinterpret_cast<uint32_t*>(smem)[i] = 0x38383838u;
  fence_proxy_async_smem();
  if (threadIdx.x == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
  if (warp == 1) tmem_alloc(&slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = slot;
  if (warp == 0) {
    if (elect_one()) {
      tmem_cp_sf(tmem + 256, umma_desc_sf(smem_u32(smem + 49152)));
      tmem_cp_sf(tmem + 260, umma_desc_sf(smem_u32(smem + 49152)));
      tmem_cp_sf(tmem + 264, umma_desc_sf(smem_u32(smem + 49152)));
    }
    __syncwarp();
    const uint64_t ad = umma_desc_sw128(smem_u32(smem)), bd = umma_desc_sw128(smem_u32(smem + 16384));
    const long long t0 = clock64();
    for (int i = 0; i < iters; i += 4) {
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if (kind == 1) umma_mxf8(tmem, ad + 2 * k, bd + 2 * k, umma_idesc_mxf8(128, N, k), tmem + 256, tmem + 260, 1);
          else umma_bf16(tmem, ad + 2 * k, bd + 2 * k, umma_idesc_bf16(128, N), 1);
        }
      }
      __syncwarp();
    }
    if (elect_one()) umma_commit(&bar);
    __syncwarp();
    mbar_wait(&bar, 0);
    const long long t1 = clock64();
    if (lane == 0) out[blockIdx.x] = t1 - t0;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

int main() {
  float* d_out;
  cudaMalloc(&d_out, 128 * 256 * sizeof(float));
  const int smem = 16384 + 256 * 128 + 3 * 512 + 1024;
  cudaFuncSetAttribute(mx_check, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  cudaFuncSetAttribute(rate, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024);
  int ok = 0;
  for (int N : {128, 256}) {
    cudaMemset(d_out, 0, 128 * 256 * sizeof(float));
    mx_check<<<1, 128, smem>>>(N, d_out);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("mx_check N=%d failed: %s\n", N, cudaGetErrorString(e)); return 1; }
    std::vector<float> h(128 * 256);
    cudaMemcpy(h.data(), d_out, h.size() * sizeof(float), cudaMemcpyDeviceToHost);
    int bad = 0;
    for (int m = 0; m < 128; ++m)
      for (int n = 0; n < N; ++n) {
        double ref = 0;
        for (int k = 0; k < 128; ++k) ref += (double)aval(m, k) * bval(n, k) * ldexp(1.0, aexp(m, k / 32) + bexp(n, k / 32));
        if (h[m * 256 + n] != (float)ref) {
          if (bad < 3) printf("  mismatch m=%d n=%d got %g want %g\n", m, n, h[m * 256 + n], ref);
          ++bad;
        }
      }
    printf("block-scaled MMA, scales by tcgen05.cp, N=%d: %s (%d mismatches)\n", N, bad ? "FAIL" : "OK", bad);
    if (!bad) ++ok;
  }
  long long* d_t;
  cudaMalloc(&d_t, 8 * sizeof(long long));
  const int iters = 4000;
  for (int kind : {0, 1})
    for (int N : {128, 256}) {
      rate<<<1, 128, 80 * 1024>>>(N, kind, iters, d_t);
      cudaError_t e = cudaDeviceSynchronize();
      if (e != cudaSuccess) { printf("rate kind %d N=%d failed: %s\n", kind, N, cudaGetErrorString(e)); return 1; }
      long long t;
      cudaMemcpy(&t, d_t, sizeof(t), cudaMemcpyDeviceToHost);
      printf("%s N=%3d: %.1f clk/MMA (K = %d per MMA)\n", kind ? "mxf8f6f4.block_scale" : "f16", N, (double)t / iters,
             kind ? 32 : 16);
    }
  return ok == 2 ? 0 : 1;
}
