// HBM-bound helper kernels of the sampling path: input assembly, posterior update, res2img,
// CLAM/SLAM gates, PIL-exact bicubic of 8- and 16-bit bands, uint8 SSE, metrics at a white level, layout conversion for
// the debug hook.
// All are coalesced/vectorised elementwise or small-reduction kernels; none needs tensor cores.
#pragma once
#include <cstdint>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include "conv_kernel.cuh"

namespace fdsr {

// ------------------------------------------------------------------------------------------
// Counter-based Gaussian noise: Philox4x32-10 keyed by the seed.  The counter is (PIXEL index inside the image,
// GLOBAL image index, stream) and one block of four normals serves up to four channels of that pixel (a second block
// serves channels 4-7, philox_pixel_normals), so the thread that owns a pixel — in particular the final conv's epilogue
// thread, which performs the posterior update in registers — needs one Philox evaluation for C <= 4.  The noise of an image depends on the seed, the
// image's index in the whole job and the step only — not on the batch it happens to be sampled in, nor on which rank
// samples it — so a batch sharded over N ranks reproduces the single-rank result bit for bit.
// Streams: T for x_T, t for the z of step t.
// Used when the caller does not inject noise (the reference draws torch.randn on the device,
// diffusion.py:189,207; any N(0,1) stream is an equally valid sample of the same sampler).
// ------------------------------------------------------------------------------------------
__global__ void set_args_kernel(SampleArgs* slot, SampleArgs a) { *slot = a; }

// x_T: the first (B,C,H,W) block of the injected noise, or stream T of the generator.  grid (HW / 256, B), thread = pixel
__global__ void noise_init_kernel(float* __restrict__ out, uint32_t HW, int C, const SampleArgs* __restrict__ args,
                                  uint32_t stream) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= HW) return;
  const size_t o = size_t(blockIdx.y) * C * HW + p;
  const float* nz = args->noise;
  float z[8];
  if (nz != nullptr) {
#pragma unroll
    for (int c = 0; c < 8; ++c) z[c] = c < C ? nz[o + size_t(c) * HW] : 0.f;
  } else {
    philox_pixel_normals(z, C, args->seed, stream, args->image0 + blockIdx.y, p);
  }
#pragma unroll
  for (int c = 0; c < 8; ++c)
    if (c < C) out[o + size_t(c) * HW] = z[c];
}

// ------------------------------------------------------------------------------------------
// Input assembly: cat([cond, x_t], 1) (diffusion.py:173) as a 16-channel NHWC 16-bit tensor
// (layout below) feeding the stem conv as a single 16-wide K chunk.
// ------------------------------------------------------------------------------------------
// Two consecutive channels of an activation tensor (16-bit packed pair, or two floats in fp32 mode)
template <typename T>
__device__ __forceinline__ float2 ld_pair(const T* p) {
  if constexpr (sizeof(T) == 4) return *reinterpret_cast<const float2*>(p);
  else return Cvt<T>::unpack(*reinterpret_cast<const uint32_t*>(p));
}
template <typename T>
__device__ __forceinline__ void st_pair(T* p, float a, float b) {
  if constexpr (sizeof(T) == 4) *reinterpret_cast<float2*>(p) = make_float2(a, b);
  else *reinterpret_cast<uint32_t*>(p) = Cvt<T>::pack(a, b);
}

// Channel order of the packed input for C bands, P = 4 if C <= 4 else 8: x_t in channels [0, C), cond in [P, P + C),
// every other channel 0 — for C = 3 [x0 x1 x2 0 | c0 c1 c2 0 | 0 x 8].  x_t comes first so that the fused posterior
// epilogue of the final conv rewrites it with one aligned store per pixel (8 bytes for P = 4, 16 for P = 8); the stem
// weights are packed with the matching permutation of the reference's cat([cond, x]) order (stem.perm in api.cu).
// One pixel of the packed input from the C x / cond channels at xp[c plane] (likewise cp); shared with the tiled
// sampler's tile_pack_kernel, whose one-tile result must equal fdsr_sample's bit for bit.
template <typename T>
__device__ __forceinline__ void pack_pixel(T* __restrict__ out, const float* __restrict__ xp,
                                           const float* __restrict__ cp, int64_t plane, int C) {
  float xv[8], cv[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    xv[c] = c < C ? xp[c * plane] : 0.f;
    cv[c] = c < C ? cp[c * plane] : 0.f;
  }
  if constexpr (sizeof(T) == 4) {
    float4* o = reinterpret_cast<float4*>(out);
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    o[0] = make_float4(xv[0], xv[1], xv[2], xv[3]);
    o[1] = C <= 4 ? make_float4(cv[0], cv[1], cv[2], cv[3]) : make_float4(xv[4], xv[5], xv[6], xv[7]);
    o[2] = C <= 4 ? z4 : make_float4(cv[0], cv[1], cv[2], cv[3]);
    o[3] = C <= 4 ? z4 : make_float4(cv[4], cv[5], cv[6], cv[7]);
  } else {
    const uint4 xs = make_uint4(Cvt<T>::pack(xv[0], xv[1]), Cvt<T>::pack(xv[2], xv[3]), Cvt<T>::pack(xv[4], xv[5]),
                                Cvt<T>::pack(xv[6], xv[7]));
    const uint4 cs = make_uint4(Cvt<T>::pack(cv[0], cv[1]), Cvt<T>::pack(cv[2], cv[3]), Cvt<T>::pack(cv[4], cv[5]),
                                Cvt<T>::pack(cv[6], cv[7]));
    uint4* o = reinterpret_cast<uint4*>(out);
    if (C <= 4) {
      o[0] = make_uint4(xs.x, xs.y, cs.x, cs.y);
      o[1] = make_uint4(0u, 0u, 0u, 0u);
    } else {
      o[0] = xs;
      o[1] = cs;
    }
  }
}

template <typename T>
__global__ void pack_input_kernel(const float* __restrict__ cond, const float* __restrict__ x,
                                  T* __restrict__ out, int B, int HW, int C) {
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (i >= int64_t(B) * HW) return;
  const int b = int(i / HW);
  const int p = int(i - int64_t(b) * HW);
  pack_pixel<T>(out + i * 16, x + int64_t(b) * C * HW + p, cond + int64_t(b) * C * HW + p, HW, C);
}

// ------------------------------------------------------------------------------------------
// Posterior update (diffusion.py:157-190), fp32, same operation order as the reference's eager
// tensor ops (no FMA contraction):
//   x0 = clamp(a*x - b*eps, -1, 1);  mean = c1*x0 + c2*x;  x_prev = mean + z*sigma
// z comes from `z` (injected) or from the Philox stream when z == nullptr and seed != nullptr.
// ------------------------------------------------------------------------------------------
// grid (HW / 256, B), thread = pixel (C channels).  z: explicit tensor (fdsr_posterior_step), else block `z_block` of
// args->noise, else the generator's stream `stream`; add_noise = 0 (t == 0): z = 0.
__global__ void posterior_kernel(const float* __restrict__ x, const float* __restrict__ eps,
                                 const float* __restrict__ z, float* __restrict__ out, uint32_t HW, int C,
                                 PostCoef k, const SampleArgs* __restrict__ args, int64_t z_block, uint32_t stream,
                                 int add_noise) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= HW) return;
  const size_t o = size_t(blockIdx.y) * C * HW + p;
  float zv[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (add_noise) {
    const float* nz = z != nullptr ? z : (args != nullptr && args->noise != nullptr
                                              ? args->noise + size_t(z_block) * gridDim.y * C * HW : nullptr);
    if (nz != nullptr) {
#pragma unroll
      for (int c = 0; c < 8; ++c)
        if (c < C) zv[c] = nz[o + size_t(c) * HW];
    } else if (args != nullptr) {
      philox_pixel_normals(zv, C, args->seed, stream, args->image0 + blockIdx.y, p);
    }
  }
#pragma unroll
  for (int c = 0; c < 8; ++c)
    if (c < C) out[o + size_t(c) * HW] = post1(x[o + size_t(c) * HW], eps[o + size_t(c) * HW], zv[c], k);
}

// res2img (diffusion.py:275-281): clamp(x,-1,1)/2 + cond.  `out` rows may be strided per sample
// so the same kernel fills the continous=True trace: out[b*out_bstride + i]; out == nullptr: frame `frame_off`
// (floats) of args->trace.  raw != 0: plain copy of x (the SR3 baseline's frames are the images themselves).
// valid != null ((B, hw) uint8, a masked tiled job): cond itself where valid is 0.
__global__ void res2img_kernel(const float* __restrict__ x, const float* __restrict__ cond,
                               float* __restrict__ out, int64_t per_sample, int64_t out_bstride,
                               int B, const SampleArgs* __restrict__ args, int64_t frame_off, int raw,
                               const uint8_t* __restrict__ valid, int64_t hw) {
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (i >= per_sample * B) return;
  float* o = out != nullptr ? out : args->trace + frame_off;
  const int64_t b = i / per_sample, r = i - b * per_sample;
  if (valid != nullptr && !valid[b * hw + r % hw]) {
    o[b * out_bstride + r] = cond[i];
    return;
  }
  const float v = fminf(fmaxf(x[i], -1.0f), 1.0f);
  o[b * out_bstride + r] = raw ? x[i] : __fadd_rn(__fdiv_rn(v, 2.0f), cond[i]);
}

// ------------------------------------------------------------------------------------------
// CLAM + SLAM gates of mid[0] (unet.py:123-173, 219-221) on a NHWC 16-bit tensor.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t f32_ordered(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ordered_f32(uint32_t u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// pool[b][c] = (sum over HW, max over HW); max kept as an order-preserving uint (memset 0 = -inf)
template <typename T>
__global__ void clam_pool_kernel(const T* __restrict__ x, unsigned long long* __restrict__ psum,
                                 uint32_t* __restrict__ pmax, int HW, int C, int pix_per_block) {
  const int b = blockIdx.y;
  const int p0 = blockIdx.x * pix_per_block;
  const int p1 = min(p0 + pix_per_block, HW);
  for (int c2 = threadIdx.x; c2 < C / 2; c2 += blockDim.x) {
    float s0 = 0.f, s1 = 0.f, m0 = -INFINITY, m1 = -INFINITY;
    const T* xp = x + (int64_t(b) * HW + p0) * C + 2 * c2;
    for (int p = p0; p < p1; ++p, xp += C) {
      const float2 f = ld_pair<T>(xp);
      s0 += f.x;
      s1 += f.y;
      m0 = fmaxf(m0, f.x);
      m1 = fmaxf(m1, f.y);
    }
    // order-independent fixed-point accumulation (bitwise reproducible)
    atomicAdd(&psum[b * C + 2 * c2], static_cast<unsigned long long>(__double2ll_rn(double(s0) * kStatScale)));
    atomicAdd(&psum[b * C + 2 * c2 + 1], static_cast<unsigned long long>(__double2ll_rn(double(s1) * kStatScale)));
    atomicMax(&pmax[b * C + 2 * c2], f32_ordered(m0));
    atomicMax(&pmax[b * C + 2 * c2 + 1], f32_ordered(m1));
  }
}

// gate[b][c] = sigmoid(W2 relu(W1 avg) + W2 relu(W1 max));  W1: [R][C], W2: [C][R]
__global__ void clam_gate_kernel(const unsigned long long* __restrict__ psum, const uint32_t* __restrict__ pmax,
                                 const float* __restrict__ w1, const float* __restrict__ w2,
                                 float* __restrict__ gate, int HW, int C, int R) {
  extern __shared__ float sm[];  // avg[C], mx[C], h[2R]
  float* avg = sm;
  float* mx = sm + C;
  float* h = sm + 2 * C;
  const int b = blockIdx.x;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    avg[c] = float(double(static_cast<long long>(psum[b * C + c])) * (1.0 / kStatScale) / double(HW));
    mx[c] = ordered_f32(pmax[b * C + c]);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
  for (int r = warp; r < 2 * R; r += nwarp) {
    const float* v = r < R ? avg : mx;
    const float* w = w1 + (r % R) * C;
    float a = 0.f;
    for (int c = lane; c < C; c += 32) a += w[c] * v[c];
    for (int o = 16; o; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) h[r] = fmaxf(a, 0.f);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float a = 0.f, m = 0.f;
    for (int r = 0; r < R; ++r) {
      a += w2[c * R + r] * h[r];
      m += w2[c * R + r] * h[R + r];
    }
    gate[b * C + c] = 1.0f / (1.0f + expf(-(a + m)));
  }
}

// sp[b][p] = (mean_c, max_c) of gate[c]*x[p][c]; one warp per pixel
template <typename T>
__global__ void slam_pool_kernel(const T* __restrict__ x, const float* __restrict__ gate,
                                 float2* __restrict__ sp, int B, int HW, int C) {
  const int64_t wid = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (wid >= int64_t(B) * HW) return;
  const int b = int(wid / HW);
  const T* xp = x + wid * C;
  const float* g = gate + b * C;
  float s = 0.f, m = -INFINITY;
  for (int c2 = lane; c2 < C / 2; c2 += 32) {
    const float2 f = ld_pair<T>(xp + 2 * c2);
    const float a = f.x * g[2 * c2], c = f.y * g[2 * c2 + 1];
    s += a + c;
    m = fmaxf(m, fmaxf(a, c));
  }
  for (int o = 16; o; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  }
  if (lane == 0) sp[wid] = make_float2(s / float(C), m);
}

// out[p][c] = sigmoid(conv7x7(sp)[p]) * gate[c] * x[p][c], plus channel-pair statistics of out.
// One warp per pixel, 8 pixels per block (256 threads); w7: [2][7][7] (avg plane, max plane).
template <typename T>
__global__ void slam_apply_kernel(const T* __restrict__ x, const float* __restrict__ gate,
                                  const float2* __restrict__ sp, const float* __restrict__ w7,
                                  T* __restrict__ out, unsigned long long* __restrict__ stats, int H, int W,
                                  int C, double sq_scale) {
  extern __shared__ float sacc[];  // [8 warps][C]: (sum, sumsq) per channel pair, one row per pixel/warp
  const int b = blockIdx.y;
  const int HW = H * W;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int p = blockIdx.x * (blockDim.x >> 5) + warp;
  float* row = sacc + warp * C;
  if (p < HW) {
    const int y = p / W, xq = p - y * W;
    float a = 0.f;
    for (int k = lane; k < 98; k += 32) {
      const int pl = k / 49, kk = k - pl * 49, ky = kk / 7, kx = kk - ky * 7;
      const int yy = y + ky - 3, xx = xq + kx - 3;
      if (yy >= 0 && yy < H && xx >= 0 && xx < W) {
        const float2 v = sp[int64_t(b) * HW + yy * W + xx];
        a += w7[k] * (pl == 0 ? v.x : v.y);
      }
    }
    for (int o = 16; o; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    const float sg = 1.0f / (1.0f + expf(-a));
    const T* xp = x + (int64_t(b) * HW + p) * C;
    T* op = out + (int64_t(b) * HW + p) * C;
    const float* g = gate + b * C;
    for (int c2 = lane; c2 < C / 2; c2 += 32) {
      const float2 f = ld_pair<T>(xp + 2 * c2);
      const float u = sg * (g[2 * c2] * f.x), v = sg * (g[2 * c2 + 1] * f.y);
      st_pair<T>(op + 2 * c2, u, v);
      row[2 * c2] = u + v;
      row[2 * c2 + 1] = u * u + v * v;
    }
  } else {
    for (int i = lane; i < C; i += 32) row[i] = 0.f;
  }
  __syncthreads();
  if (stats != nullptr)
    for (int i = threadIdx.x; i < C; i += blockDim.x) {
      float t = 0.f;
      for (int w8 = 0; w8 < 8; ++w8) t += sacc[w8 * C + i];  // fixed order
      atomicAdd(&stats[int64_t(b) * C + i],   // [pair][2]: even = sum, odd = sum of squares
                static_cast<unsigned long long>(__double2ll_rn(double(t) * ((i & 1) ? sq_scale : kStatScale))));
    }
}

// ------------------------------------------------------------------------------------------
// PIL-exact bicubic (Pillow ImagingResample, 8 bpc): separable, horizontal first, 22-bit fixed
// point taps, uint8 rounding + clipping after each pass.  bounds/taps are built on the host.
// ------------------------------------------------------------------------------------------
constexpr int kBicPrec = 22;
// C <= 8 bands, each resized on its own exactly as Pillow resizes one 8-bit band.
// in: [B][inH][inW][C] u8 -> out: [B][inH][outW][C] u8
__global__ void bicubic_h_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out,
                                 const int* __restrict__ xmin, const int* __restrict__ xcnt,
                                 const int* __restrict__ taps, int ksize, int B, int inH, int inW, int outW, int C) {
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  const int64_t total = int64_t(B) * inH * outW;
  if (i >= total) return;
  const int xo = int(i % outW);
  const int64_t row = i / outW;
  const uint8_t* src = in + (row * inW + xmin[xo]) * C;
  const int* k = taps + xo * ksize;
  int a[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) a[c] = 1 << (kBicPrec - 1);
  for (int j = 0; j < xcnt[xo]; ++j)
#pragma unroll
    for (int c = 0; c < 8; ++c)
      if (c < C) a[c] += int(src[C * j + c]) * k[j];
  uint8_t* o = out + i * C;
#pragma unroll
  for (int c = 0; c < 8; ++c)
    if (c < C) o[c] = uint8_t(min(max(a[c] >> kBicPrec, 0), 255));
}
// in: [B][inH][W][C] u8 -> out_u8: [B][outH][W][C] (optional), cond: [B][C][outH][W] fp32 (optional)
__global__ void bicubic_v_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out_u8,
                                 float* __restrict__ cond, const int* __restrict__ ymin,
                                 const int* __restrict__ ycnt, const int* __restrict__ taps, int ksize,
                                 int B, int inH, int outH, int W, int C) {
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  const int64_t total = int64_t(B) * outH * W;
  if (i >= total) return;
  const int x = int(i % W);
  const int yo = int((i / W) % outH);
  const int b = int(i / (int64_t(W) * outH));
  const uint8_t* src = in + ((int64_t(b) * inH + ymin[yo]) * W + x) * C;
  const int* k = taps + yo * ksize;
  int a[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) a[c] = 1 << (kBicPrec - 1);
  for (int j = 0; j < ycnt[yo]; ++j) {
    const uint8_t* s = src + int64_t(j) * W * C;
#pragma unroll
    for (int c = 0; c < 8; ++c)
      if (c < C) a[c] += int(s[c]) * k[j];
  }
  const int64_t plane = int64_t(outH) * W;
  float* cp = cond != nullptr ? cond + int64_t(b) * C * plane + int64_t(yo) * W + x : nullptr;
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    if (c >= C) continue;
    const int v = min(max(a[c] >> kBicPrec, 0), 255);
    if (out_u8 != nullptr) out_u8[i * C + c] = uint8_t(v);
    // ToTensor (/255) then *2-1 (data/util.py:66-75), fp32, same operation order
    if (cp != nullptr) cp[c * plane] = __fsub_rn(__fmul_rn(__fdiv_rn(float(v), 255.0f), 2.0f), 1.0f);
  }
}

// ------------------------------------------------------------------------------------------
// PIL-exact bicubic of 16-bit bands (Pillow ImagingResample of an 'I;16' image): the same bounds as the 8-bit pair and
// the normalised double weights before their fixed-point step; per output sample ss = 0.0, ss = ss + double(p) * k[j]
// with every multiply and add rounded on its own (no FMA contraction), rounded half away from zero, then stored the
// way Pillow stores an I;16 sample byte by byte: lo = CLIP8(v % 256), hi = CLIP8(v >> 8).  So v < 0 -> 0 and
// v > 65535 -> 65280 + v % 256 (not 65535).  The horizontal pass's result is stored the same way (uint16 intermediate).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint16_t pil_store_u16(double ss) {
  const int v = int(ss >= 0.0 ? floor(__dadd_rn(ss, 0.5)) : -floor(__dadd_rn(-ss, 0.5)));
  if (v < 0) return 0;
  if (v > 65535) return uint16_t(0xff00 | (v & 0xff));
  return uint16_t(v);
}
// in: [B][inH][inW][C] u16 -> out: [B][inH][outW][C] u16
__global__ void bicubic16_h_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out,
                                   const int* __restrict__ xmin, const int* __restrict__ xcnt,
                                   const double* __restrict__ wts, int ksize, int B, int inH, int inW, int outW,
                                   int C) {
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  const int64_t total = int64_t(B) * inH * outW;
  if (i >= total) return;
  const int xo = int(i % outW);
  const int64_t row = i / outW;
  const uint16_t* src = in + (row * inW + xmin[xo]) * C;
  const double* k = wts + xo * ksize;
  double a[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) a[c] = 0.0;
  for (int j = 0; j < xcnt[xo]; ++j) {
    const double kj = k[j];
#pragma unroll
    for (int c = 0; c < 8; ++c)
      if (c < C) a[c] = __dadd_rn(a[c], __dmul_rn(double(src[C * j + c]), kj));
  }
  uint16_t* o = out + i * C;
#pragma unroll
  for (int c = 0; c < 8; ++c)
    if (c < C) o[c] = pil_store_u16(a[c]);
}
// in: [B][inH][W][C] u16 -> out_u16: [B][outH][W][C] (optional, the stored levels), cond: [B][C][outH][W] fp32
// (optional) = (min(v, M) / M) * 2 - 1 in fp32, the operation order of the 8-bit pass with 255 -> M
__global__ void bicubic16_v_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out_u16,
                                   float* __restrict__ cond, const int* __restrict__ ymin,
                                   const int* __restrict__ ycnt, const double* __restrict__ wts, int ksize,
                                   int B, int inH, int outH, int W, int C, int M) {
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  const int64_t total = int64_t(B) * outH * W;
  if (i >= total) return;
  const int x = int(i % W);
  const int yo = int((i / W) % outH);
  const int b = int(i / (int64_t(W) * outH));
  const uint16_t* src = in + ((int64_t(b) * inH + ymin[yo]) * W + x) * C;
  const double* k = wts + yo * ksize;
  double a[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) a[c] = 0.0;
  for (int j = 0; j < ycnt[yo]; ++j) {
    const uint16_t* s = src + int64_t(j) * W * C;
    const double kj = k[j];
#pragma unroll
    for (int c = 0; c < 8; ++c)
      if (c < C) a[c] = __dadd_rn(a[c], __dmul_rn(double(s[c]), kj));
  }
  const int64_t plane = int64_t(outH) * W;
  float* cp = cond != nullptr ? cond + int64_t(b) * C * plane + int64_t(yo) * W + x : nullptr;
  const float fM = float(M);
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    if (c >= C) continue;
    const int v = pil_store_u16(a[c]);
    if (out_u16 != nullptr) out_u16[i * C + c] = uint16_t(v);
    if (cp != nullptr) cp[c * plane] = __fsub_rn(__fmul_rn(__fdiv_rn(float(min(v, M)), fM), 2.0f), 1.0f);
  }
}

// ------------------------------------------------------------------------------------------
// Sum of squared uint8 differences per image after tensor2img quantisation (core/metrics.py:16-42)
// ------------------------------------------------------------------------------------------
// tensor2img at white level M: the level 0..M of an fp32 value in [-1, 1]
__device__ __forceinline__ int quant_level(float v, float M) {
  v = fminf(fmaxf(v, -1.0f), 1.0f);
  v = __fdiv_rn(__fadd_rn(v, 1.0f), 2.0f);
  return __float2int_rn(__fmul_rn(v, M));  // numpy .round(): half to even
}
__device__ __forceinline__ int quant_u8(float v) { return quant_level(v, 255.0f); }
__global__ void sse_u8_kernel(const float* __restrict__ a, const float* __restrict__ b,
                              double* __restrict__ sse, int64_t per_image) {
  const int img = blockIdx.y;
  const float* ap = a + img * per_image;
  const float* bp = b + img * per_image;
  unsigned long long acc = 0;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < per_image;
       i += int64_t(gridDim.x) * blockDim.x) {
    const int d = quant_u8(ap[i]) - quant_u8(bp[i]);
    acc += (unsigned long long)(d * d);
  }
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0 && acc) atomicAdd(&sse[img], double(acc));
}

// ------------------------------------------------------------------------------------------
// Evaluation metrics of sr_mfe.py:315-345 on tensor2img-quantised images at white level M (255: uint8), per image:
//   acc[b][0] = sum (a-b)^2            (compare_mse / compare_psnr / calculate_ergas)
//   acc[b][1] = sum a                  (calculate_ergas: mean of the first image)
//   acc[b][2] = sum of the SSIM map over the cropped interior and the C channels, 2^-40 fixed point
// SSIM follows skimage.measure.compare_ssim(X, Y, multichannel=True) as the reference calls it
// (scikit-image 0.15, _structural_similarity.py): 7x7 uniform window, K1 = 0.01, K2 = 0.03,
// data_range = M, sample covariance (x 49/48), float64, mean over the map cropped by 3 pixels per
// side, then mean over channels.  Window sums are exact integers (int64: 49 * 65535^2 > 2^31); the map is evaluated
// in fp64.  M = 255 computes exactly what the uint8 form of this kernel computed.
// Masked (fdsr_metrics_masked, valid = (B,H,W) uint8): the three sums run over the valid pixels and over the windows
// whose 49 pixels are all valid, and
//   acc[b][3] = number of valid values (C |V|),  acc[b][4] = number of SSIM map entries summed (over the C channels).
// ------------------------------------------------------------------------------------------
constexpr int kSsimWin = 7, kSsimPad = 3, kSsimTile = 16;
constexpr int kMetricSlots = 8;  // accumulators per image
constexpr double kSsimScale = 1099511627776.0;  // 2^40

__global__ void __launch_bounds__(256) metrics_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                      unsigned long long* __restrict__ acc, int H, int W, int C,
                                                      int M, const uint8_t* __restrict__ valid) {
  __shared__ uint16_t sa[kSsimTile + 6][kSsimTile + 6 + 2], sb[kSsimTile + 6][kSsimTile + 6 + 2];
  __shared__ uint8_t sv[kSsimTile + 6][kSsimTile + 6 + 2];
  __shared__ long long red[8][5];
  const int img = blockIdx.z / C, ch = blockIdx.z % C;  // grid z = B * C
  const float* ap = a + (int64_t(img) * C + ch) * H * W;
  const float* bp = b + (int64_t(img) * C + ch) * H * W;
  const float fM = float(M);
  // the block owns the 16x16 pixels at (y0, x0); its SSIM windows need a 3-pixel apron
  const int y0 = blockIdx.y * kSsimTile, x0 = blockIdx.x * kSsimTile;
  for (int e = threadIdx.x; e < (kSsimTile + 6) * (kSsimTile + 6); e += 256) {
    const int ly = e / (kSsimTile + 6), lx = e - ly * (kSsimTile + 6);
    const int y = y0 + ly - kSsimPad, x = x0 + lx - kSsimPad;
    const bool in = y >= 0 && y < H && x >= 0 && x < W;
    sa[ly][lx] = in ? uint16_t(quant_level(ap[int64_t(y) * W + x], fM)) : 0;
    sb[ly][lx] = in ? uint16_t(quant_level(bp[int64_t(y) * W + x], fM)) : 0;
    if (valid != nullptr) sv[ly][lx] = in && valid[(int64_t(img) * H + y) * W + x] != 0;
  }
  __syncthreads();
  const int ly = threadIdx.x / kSsimTile, lx = threadIdx.x % kSsimTile;
  const int y = y0 + ly, x = x0 + lx;
  long long sse = 0, suma = 0, ss = 0, nv = 0, nw = 0;
  if (y < H && x < W && (valid == nullptr || sv[ly + kSsimPad][lx + kSsimPad])) {
    const int va = sa[ly + kSsimPad][lx + kSsimPad], vb = sb[ly + kSsimPad][lx + kSsimPad];
    sse = (long long)(va - vb) * (va - vb);
    suma = va;
    nv = 1;
    bool win = y >= kSsimPad && y < H - kSsimPad && x >= kSsimPad && x < W - kSsimPad;
    if (win && valid != nullptr) {
#pragma unroll
      for (int dy = 0; dy < kSsimWin; ++dy)
#pragma unroll
        for (int dx = 0; dx < kSsimWin; ++dx) win = win && sv[ly + dy][lx + dx];
    }
    if (win) {
      nw = 1;
      int s1 = 0, s2 = 0;
      long long s11 = 0, s22 = 0, s12 = 0;
#pragma unroll
      for (int dy = 0; dy < kSsimWin; ++dy)
#pragma unroll
        for (int dx = 0; dx < kSsimWin; ++dx) {
          const unsigned p = sa[ly + dy][lx + dx], q = sb[ly + dy][lx + dx];
          s1 += p;
          s2 += q;
          s11 += p * p;
          s22 += q * q;
          s12 += p * q;
        }
      const double np = double(kSsimWin * kSsimWin), cov = np / (np - 1.0);
      const double ux = s1 / np, uy = s2 / np;
      const double vx = cov * (s11 / np - ux * ux), vy = cov * (s22 / np - uy * uy), vxy = cov * (s12 / np - ux * uy);
      // C1, C2 rounded on their own, as the compile-time constants of M = 255 were (an FMA would fuse their last
      // multiply into the sums below and change the bits)
      const double R = double(M), C1 = __dmul_rn(0.01 * R, 0.01 * R), C2 = __dmul_rn(0.03 * R, 0.03 * R);
      const double S = ((2.0 * ux * uy + C1) * (2.0 * vxy + C2)) / ((ux * ux + uy * uy + C1) * (vx + vy + C2));
      ss = __double2ll_rn(S * kSsimScale);
    }
  }
  for (int o = 16; o; o >>= 1) {
    sse += __shfl_xor_sync(0xffffffffu, sse, o);
    suma += __shfl_xor_sync(0xffffffffu, suma, o);
    ss += __shfl_xor_sync(0xffffffffu, ss, o);
    nv += __shfl_xor_sync(0xffffffffu, nv, o);
    nw += __shfl_xor_sync(0xffffffffu, nw, o);
  }
  const int warp = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) {
    red[warp][0] = sse;
    red[warp][1] = suma;
    red[warp][2] = ss;
    red[warp][3] = nv;
    red[warp][4] = nw;
  }
  __syncthreads();
  if (threadIdx.x < 5) {
    long long t = 0;
    for (int w8 = 0; w8 < 8; ++w8) t += red[w8][threadIdx.x];
    if (t) atomicAdd(&acc[img * kMetricSlots + threadIdx.x], static_cast<unsigned long long>(t));  // order-independent
  }
}

// out[b] = (mse, psnr, ssim, ergas) in float64, exactly as sr_mfe.py derives them from the sums (C bands: n = C H W,
// SSIM averaged over the C channels, ERGAS divided by C); PSNR = 10 log10(M^2 / mse).  masked: n and the SSIM
// divisor are the counts acc[b][3] and acc[b][4]; no valid value gives four NaNs, no whole valid window a NaN SSIM.
// With every pixel valid the counts equal C H W and C (H-6) (W-6), so the result is the unmasked one bit for bit.
__global__ void metrics_finalize_kernel(const unsigned long long* __restrict__ acc, double* __restrict__ out, int B,
                                        int H, int W, int C, double scale, int M, int masked) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const unsigned long long* ab = acc + b * kMetricSlots;
  const double n = masked ? double(static_cast<long long>(ab[3])) : double(C) * H * W;
  if (n == 0.0) {
    out[b * 4 + 0] = out[b * 4 + 1] = out[b * 4 + 2] = out[b * 4 + 3] = NAN;
    return;
  }
  const double sse = double(static_cast<long long>(ab[0]));
  const double mean = double(static_cast<long long>(ab[1])) / n;
  const double mse = sse / n;
  const double nss = masked ? double(static_cast<long long>(ab[4]))
                            : double(C) * double(H - 2 * kSsimPad) * double(W - 2 * kSsimPad);
  out[b * 4 + 0] = mse;
  out[b * 4 + 1] = mse > 0.0 ? 10.0 * log10(double(M) * double(M) / mse) : INFINITY;
  out[b * 4 + 2] = (masked ? nss > 0.0 : (H > 2 * kSsimPad && W > 2 * kSsimPad))
                       ? double(static_cast<long long>(ab[2])) / kSsimScale / nss : NAN;
  out[b * 4 + 3] = 100.0 * sqrt(mse / (mean * mean) / double(C)) / scale;
}

// NHWC 16-bit -> NCHW fp32 (debug hook only)
template <typename T>
__global__ void nhwc_to_nchw_kernel(const T* __restrict__ in, float* __restrict__ out, int B, int HW, int C) {
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (i >= int64_t(B) * HW * C) return;
  const int c = int(i % C);
  const int64_t bp = i / C;
  const int b = int(bp / HW);
  const int p = int(bp - int64_t(b) * HW);
  float v;
  if constexpr (sizeof(T) == 4) v = in[i];
  else if constexpr (Cvt<T>::kFmt == 0) v = __half2float(in[i]);
  else v = __bfloat162float(in[i]);
  out[(int64_t(b) * C + c) * HW + p] = v;
}

}  // namespace fdsr
