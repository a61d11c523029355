// Philox4x32-10 dropout stream shared by every dropout kernel of the library (train_ops.cu: avh_dropout and the
// no-grad training forward; train_dropout.cu: the training step's forward and backward).
// Element i of a site's tensor ([rows, C] row-major) takes lane i % 4 of philox4x32(seed, i / 4, site) and is kept
// when u01(lane) >= p, scaled by 1 / (1 - p).  That mapping is what makes a forward, its backward and avh_dropout
// agree bit for bit, so it lives here only.
#pragma once

namespace avh {

// counter = (element block, site), key = seed (Salmon et al., SC'11)
__device__ __forceinline__ uint4 philox4x32(unsigned long long seed, unsigned long long ctr_lo, unsigned int site) {
  unsigned int k0 = (unsigned int)seed, k1 = (unsigned int)(seed >> 32);
  unsigned int c0 = (unsigned int)ctr_lo, c1 = (unsigned int)(ctr_lo >> 32), c2 = site, c3 = 0x5eedu;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const unsigned int hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const unsigned int hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const unsigned int n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ float u01(unsigned int x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }

// the four mask values (0 or 1 / (1 - p)) of elements 4 * blk .. 4 * blk + 3
__device__ __forceinline__ float4 dropout_mask4(unsigned long long seed, long long blk, unsigned int site, float p) {
  const uint4 r = philox4x32(seed, (unsigned long long)blk, site);
  const float keep = 1.f / (1.f - p);
  return make_float4(u01(r.x) >= p ? keep : 0.f, u01(r.y) >= p ? keep : 0.f, u01(r.z) >= p ? keep : 0.f,
                     u01(r.w) >= p ? keep : 0.f);
}

}  // namespace avh
