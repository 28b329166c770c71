// Tiled sampling of canvases of any size (fdsr_sample_tiled, include/fdsr.h; DESIGN §4.4): overlapping tiles share
// one canvas-wide chain.  Every step, the tiles' eps predictions are blended into one canvas-wide eps and a single
// posterior update moves the canvas-wide x_t (MultiDiffusion in eps space).
//
// Grid rule per axis (length L, tile t, overlap o):  t_e = min(t, 8 floor(L/8)), o_e = min(o, t_e - 8), s = t_e - o_e;
// starts i*s for every i with i*s < L - t_e, then L - t_e (the last tile is flush with the far edge).
// Weight of tile offset i: r(i) = min(i + 1, t_e - i, o_e + 1); a tile pixel weighs r_y * r_x (an exact integer).
#pragma once
#include <cstdint>
#include "aux_kernels.cuh"

namespace fdsr {

struct TileAxis {
  int32_t L;   // canvas extent
  int32_t te;  // effective tile extent (multiple of 8, <= L)
  int32_t oe;  // effective overlap
  int32_t s;   // stride te - oe (>= 8)
  int32_t n;   // tiles on this axis: starts i*s for i < n - 1, then L - te
};

__host__ __device__ __forceinline__ int tile_start(const TileAxis& a, int i) { return i + 1 < a.n ? i * a.s : a.L - a.te; }
__host__ __device__ __forceinline__ int tile_ramp(const TileAxis& a, int i) {
  return min(min(i + 1, a.te - i), a.oe + 1);
}

// Tiles of one axis covering position y, in ascending start order: the regular tiles lo..hi, then the flush last tile
// n - 1 when it covers y (it starts after every regular tile, so the order is the global one).
struct TileCover {
  int lo, cnt_reg, last;  // last = n - 1 or -1
  __device__ __forceinline__ int count() const { return cnt_reg + (last >= 0 ? 1 : 0); }
  __device__ __forceinline__ int at(int k) const { return k < cnt_reg ? lo + k : last; }
};
__device__ __forceinline__ TileCover tile_cover(const TileAxis& a, int y) {
  const int d = y - a.te + 1;
  const int lo = d <= 0 ? 0 : (d + a.s - 1) / a.s;
  const int hi = min(y / a.s, a.n - 2);
  TileCover c;
  c.lo = lo;
  c.cnt_reg = hi >= lo ? hi - lo + 1 : 0;
  c.last = y >= a.L - a.te ? a.n - 1 : -1;
  return c;
}

// Tile activity of a masked job (fdsr_sample_tiled_masked): flags[g] = 1 iff the window of global tile g holds a
// pixel with valid != 0.  valid: (B,H,W) uint8.  grid n_tiles, one block per tile.
__global__ void __launch_bounds__(256) tile_active_kernel(const uint8_t* __restrict__ valid, TileAxis ay, TileAxis ax,
                                                          uint8_t* __restrict__ flags) {
  const int64_t g = blockIdx.x, per_canvas = int64_t(ay.n) * ax.n;
  const int64_t b = g / per_canvas;
  const int r = int(g - b * per_canvas);
  const int y0 = tile_start(ay, r / ax.n), x0 = tile_start(ax, r % ax.n);
  const uint8_t* v = valid + b * int64_t(ay.L) * ax.L + int64_t(y0) * ax.L + x0;
  int any = 0;
  for (int p = threadIdx.x; p < ay.te * ax.te && !any; p += blockDim.x) {
    const int py = p / ax.te;
    any = v[int64_t(py) * ax.L + (p - py * ax.te)] != 0;
  }
  any = __syncthreads_or(any);
  if (threadIdx.x == 0) flags[g] = uint8_t(any);
}

// Packed 16-channel NHWC network input of one chunk of `bc` tiles (x_t and cond of C bands, pack_pixel), read
// from the canvases at each tile's window.  Chunk slot j holds tile slot min(tile0 + j, g_last), g_last = the last
// slot of the caller's own range: its last chunk is padded with repeats of that slot.  Slot s is global tile act[s]
// (the active tiles of a masked job), or s itself when act is null.  One thread per tile pixel.
template <typename T>
__global__ void tile_pack_kernel(const float* __restrict__ cond, const float* __restrict__ x, T* __restrict__ out,
                                 TileAxis ay, TileAxis ax, int64_t tile0, int64_t g_last, int bc, int C,
                                 const int64_t* __restrict__ act) {
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  const int64_t tpx = int64_t(ay.te) * ax.te;
  if (i >= bc * tpx) return;
  const int64_t j = i / tpx;
  const int p = int(i - j * tpx);
  const int64_t s = min(tile0 + j, g_last);
  const int64_t g = act != nullptr ? act[s] : s;
  const int64_t per_canvas = int64_t(ay.n) * ax.n;
  const int64_t b = g / per_canvas;
  const int r = int(g - b * per_canvas);
  const int py = p / ax.te, px = p - py * ax.te;
  const int y = tile_start(ay, r / ax.n) + py, xx = tile_start(ax, r % ax.n) + px;
  const int64_t plane = int64_t(ay.L) * ax.L;
  const int64_t o = b * C * plane + int64_t(y) * ax.L + xx;
  pack_pixel<T>(out + i * 16, x + o, cond + o, plane, C);
}

// The covering tiles of one axis form one contiguous index range: the regular tiles cover [0, (n-2) s + t_e) without
// gaps (s <= t_e), and the flush last tile starts at L - t_e <= (n-1) s, so a position it covers is covered by tile n-2
// or by no regular tile.  Hence the covering tiles of a pixel are a rectangle [cy.at(0), cy.at(ny-1)] x
// [cx.at(0), cx.at(nx-1)] of the tile grid, and its first covering tile in global order is (cy.at(0), cx.at(0)).
__device__ __forceinline__ int64_t tile_row_base(const TileAxis& ay, const TileAxis& ax, int b, int ty) {
  return (int64_t(b) * ay.n + ty) * ax.n;
}

// One step on the canvases: eps of each pixel = the normalised-weight blend of the eps of the tiles covering it (global
// tile order, fp32, round-to-nearest, the sum starting from the first term so that a pixel covered once gets its tile's
// eps exactly), then x_{t-1} = post1(x_t, eps, z) in place.  z: block z_block of args->noise, else the generator's
// stream `stream` at (image0 + canvas, pixel index y*W + x); add_noise = 0 (t == 0): z = 0.  No atomics: each thread
// owns its pixel.  x: (B,C,H,W); eps_store: [slot][C][te_y][te_x], global tile g in slot slot[g], or in slot g when
// slot is null.  A masked job's inactive tiles (slot -1) are left out of both sums, so "first" is the first active
// term; a pixel with no active covering tile is not updated.
// Own range [g0, g1): a pixel is updated iff one of its covering tiles lies in it (the union of the own tiles' windows,
// fdsr_sample_tiled_part); [0, n_tiles) updates every pixel.  grid (ceil((p1 - p0) / 256), canvases): canvas
// b0 + blockIdx.y, pixel indices [p0, p1) of it -- a band that contains every pixel the range updates.
__global__ void tile_blend_posterior_kernel(float* __restrict__ x, const float* __restrict__ eps_store, TileAxis ay,
                                            TileAxis ax, int C, PostCoef k, const SampleArgs* __restrict__ args,
                                            int64_t z_block, uint32_t stream, int add_noise, int B, int b0, uint32_t p0,
                                            uint32_t p1, int64_t g0, int64_t g1, const int32_t* __restrict__ slot) {
  const uint32_t HW = uint32_t(ay.L) * uint32_t(ax.L);
  const uint32_t p = p0 + blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= p1) return;
  const int b = b0 + blockIdx.y;
  const int y = int(p / uint32_t(ax.L)), xx = int(p - uint32_t(y) * uint32_t(ax.L));
  const TileCover cy = tile_cover(ay, y), cx = tile_cover(ax, xx);
  const int ny = cy.count(), nx = cx.count();
  bool own = false;
  for (int a = 0; a < ny; ++a) {
    const int64_t r = tile_row_base(ay, ax, b, cy.at(a));
    own |= r + cx.at(nx - 1) >= g0 && r + cx.at(0) < g1;
  }
  if (!own) return;
  float wsum = 0.f;
  bool any = false;
  for (int a = 0; a < ny; ++a) {
    const int ry = tile_ramp(ay, y - tile_start(ay, cy.at(a)));
    const int64_t r = tile_row_base(ay, ax, b, cy.at(a));
    for (int c = 0; c < nx; ++c) {
      if (slot != nullptr && slot[r + cx.at(c)] < 0) continue;
      const float w = float(ry * tile_ramp(ax, xx - tile_start(ax, cx.at(c))));
      wsum = any ? __fadd_rn(wsum, w) : w;
      any = true;
    }
  }
  if (!any) return;
  const int64_t tpx = int64_t(ay.te) * ax.te;
  float e[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  bool first = true;
  for (int a = 0; a < ny; ++a) {
    const int ty = cy.at(a), oy = y - tile_start(ay, ty);
    const int ry = tile_ramp(ay, oy);
    for (int c = 0; c < nx; ++c) {
      const int tx = cx.at(c), ox = xx - tile_start(ax, tx);
      const int64_t g = tile_row_base(ay, ax, b, ty) + tx;
      const int64_t sg = slot != nullptr ? int64_t(slot[g]) : g;
      if (sg < 0) continue;
      const float nk = __fdiv_rn(float(ry * tile_ramp(ax, ox)), wsum);
      const float* ep = eps_store + sg * C * tpx + int64_t(oy) * ax.te + ox;
#pragma unroll
      for (int ch = 0; ch < 8; ++ch) {
        if (ch >= C) continue;
        const float term = __fmul_rn(nk, ep[ch * tpx]);
        e[ch] = first ? term : __fadd_rn(e[ch], term);
      }
      first = false;
    }
  }
  const size_t o = size_t(b) * C * HW + p;
  float zv[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (add_noise) {
    if (args->noise != nullptr) {
      const float* nz = args->noise + size_t(z_block) * B * C * HW;
#pragma unroll
      for (int ch = 0; ch < 8; ++ch)
        if (ch < C) zv[ch] = nz[o + size_t(ch) * HW];
    } else {
      philox_pixel_normals(zv, C, args->seed, stream, args->image0 + b, p);
    }
  }
#pragma unroll
  for (int ch = 0; ch < 8; ++ch)
    if (ch < C) x[o + size_t(ch) * HW] = post1(x[o + size_t(ch) * HW], e[ch], zv[ch], k);
}

// res2img_kernel restricted to the pixels whose first covering tile (global order) lies in [g0, g1): those get
// clamp(x,-1,1)/2 + cond, every other pixel +0.0, so an integer sum of the bit patterns written by ranks whose ranges
// partition the tiles rebuilds the whole image.  out[b*out_bstride + ch*HW + p]; out == nullptr: frame `frame_off`
// (floats) of args->trace.  grid (ceil(HW / 256), B), thread = pixel.
__global__ void res2img_owned_kernel(const float* __restrict__ x, const float* __restrict__ cond,
                                     float* __restrict__ out, int64_t out_bstride, int C, TileAxis ay, TileAxis ax,
                                     int64_t g0, int64_t g1, const SampleArgs* __restrict__ args, int64_t frame_off) {
  const uint32_t HW = uint32_t(ay.L) * uint32_t(ax.L);
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= HW) return;
  const int b = blockIdx.y;
  const int y = int(p / uint32_t(ax.L)), xx = int(p - uint32_t(y) * uint32_t(ax.L));
  const int64_t g = tile_row_base(ay, ax, b, tile_cover(ay, y).at(0)) + tile_cover(ax, xx).at(0);
  const bool own = g >= g0 && g < g1;
  float* o = (out != nullptr ? out : args->trace + frame_off) + b * out_bstride + p;
  const size_t i = size_t(b) * C * HW + p;
  for (int ch = 0; ch < C; ++ch) {
    const float v = fminf(fmaxf(x[i + size_t(ch) * HW], -1.0f), 1.0f);
    o[size_t(ch) * HW] = own ? __fadd_rn(__fdiv_rn(v, 2.0f), cond[i + size_t(ch) * HW]) : 0.0f;
  }
}

}  // namespace fdsr
