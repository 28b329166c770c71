// Arithmetic shared by the sampler's stand-alone kernels (aux_kernels.cuh) and the fused posterior epilogue of the
// final conv (conv_kernel.cuh): the counter-based Gaussian generator and the p_sample update.
#pragma once
#include <cstdint>
#include "conv_desc.h"

namespace fdsr {

__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += 0x9E3779B9u;
    key.y += 0xBB67AE85u;
  }
  return ctr;
}
// `flip` is XORed into the fourth counter word: 0 for block 0 of a pixel, 0x80000000 for block 1
__device__ __forceinline__ float4 philox_normal4(uint64_t seed, uint32_t stream, uint64_t image, uint32_t idx4,
                                                 uint32_t flip = 0u) {
  const uint4 r = philox4x32_10(make_uint4(idx4, uint32_t(image), stream, (0x5eedu + uint32_t(image >> 32)) ^ flip),
                                make_uint2(uint32_t(seed), uint32_t(seed >> 32)));
  const float k = 2.3283064365386963e-10f;  // 2^-32
  const float u0 = (float(r.x) + 0.5f) * k, u1 = (float(r.y) + 0.5f) * k;
  const float u2 = (float(r.z) + 0.5f) * k, u3 = (float(r.w) + 0.5f) * k;
  const float r0 = sqrtf(-2.0f * __logf(u0)), r1 = sqrtf(-2.0f * __logf(u2));
  float s0, c0, s1, c1;
  __sincosf(6.283185307179586f * u1, &s0, &c0);
  __sincosf(6.283185307179586f * u3, &s1, &c1);
  return make_float4(r0 * c0, r0 * s0, r1 * c1, r1 * s1);
}

// Built-in noise of one pixel of a C-band image (C <= 8; include/fdsr.h, fdsr_set_image_offset): channel c takes
// normal c mod 4 of Philox block c div 4.  Block 1 is only evaluated for C > 4, so C <= 4 costs one block.
__device__ __forceinline__ void philox_pixel_normals(float (&z)[8], int C, uint64_t seed, uint32_t stream,
                                                     uint64_t image, uint32_t pixel) {
  const float4 a = philox_normal4(seed, stream, image, pixel);
  z[0] = a.x;
  z[1] = a.y;
  z[2] = a.z;
  z[3] = a.w;
  if (C > 4) {
    const float4 b = philox_normal4(seed, stream, image, pixel, 0x80000000u);
    z[4] = b.x;
    z[5] = b.y;
    z[6] = b.z;
    z[7] = b.w;
  } else {
    z[4] = z[5] = z[6] = z[7] = 0.f;
  }
}

// Posterior update (diffusion.py:157-190), fp32, same operation order as the reference's eager tensor ops (no FMA
// contraction):  x0 = clamp(a*x - b*eps, -1, 1);  mean = c1*x0 + c2*x;  x_prev = mean + z*sigma
__device__ __forceinline__ float post1(float x, float e, float z, const PostCoef& k) {
  float x0 = __fsub_rn(__fmul_rn(k.a, x), __fmul_rn(k.b, e));
  x0 = fminf(fmaxf(x0, -1.0f), 1.0f);
  const float mean = __fadd_rn(__fmul_rn(k.c1, x0), __fmul_rn(k.c2, x));
  return __fadd_rn(mean, __fmul_rn(z, k.sigma));
}

}  // namespace fdsr
