// conv_gemm_kernel: the one heavy kernel of the sampling path (sm_100a only).
//
// Implicit-GEMM convolution on tcgen05 tensor cores with fp32 accumulators in TMEM:
//   M = 256 output pixels per CTA tile (32x8 pixels = two 128-row MMA tiles), N = all output
//   channels (16/64/128/256), K = taps x input channels, walked in chunks of 64 channels.
//
// Warp roles (640 threads, 1 CTA / SM, persistent over a contiguous range of tiles):
//   warp 0      MMA issuer (one elected thread): tcgen05.mma from shared-memory descriptors
//   warp 1      loader (one elected thread): TMA tensor loads of the input patches (one per 64-channel
//               chunk, 128B-swizzled, zero-filled halo) and cp.async.bulk of pre-packed weight tap blobs
//   warps 4-11  epilogue (one warpgroup per 128-row MMA tile): tcgen05.ld -> bias/FiLM -> residual
//               -> 16-bit TMA store -> GroupNorm pair statistics
//   warps 2,3,12-19  producers: GroupNorm scale/shift + Swish applied in place to the TMA-delivered
//               patch (pixel-major, 128 B per position); for the nine-tap nearest-upsample convs
//               coalesced 16B global loads of the 2x-upsampled patch, 16B stores into a no-swizzle
//               [channel group][position][8 ch] patch.
// The patch is loaded and transformed ONCE per 64-channel chunk and then serves all nine 3x3
// taps as shifted shared-memory descriptor views (start address + 128 B * (dy*10 + dx), SBO =
// 1280 B; the MMA unit swizzles on absolute address bits, tools/probe_umma.cu), so the A operand is
// never re-fetched per tap and GroupNorm/Swish/concat/upsample/space-to-depth never touch HBM as
// separate passes.
//
// The kernel is instruction-issue sensitive (ncu: ~0.45 IPC per scheduler with 5 warps each), so
// the layer description is a __grid_constant__ kernel parameter (constant-bank operands instead of
// shared-memory loads), waits use the mbarrier suspend hint instead of spinning, and for N = 64 the
// GroupNorm statistics are kept as per-lane running sums in spare TMEM columns and reduced across
// lanes only once per tile group.
//
// Reference ops covered (FastDiffSR/model/fastdiffsr_modules/unet.py): Block :89-101 (GroupNorm,
// Swish, Conv3x3), ResnetBlock :104-120 (FiLM add, residual 1x1 / identity), Downsample :77-83,
// Upsample :66-74, the skip concatenation :317-321, stem :257-258 and final_conv :297.
#pragma once
#include "conv_desc.h"
#include "ptx.cuh"
#include "sampler_math.cuh"

namespace fdsr {

constexpr int kConvThreads = 640;              // 20 warps = 5 per scheduler (register file: 96 regs/thread)
constexpr int kProdWarps = 10;
constexpr int kProdThreads = kProdWarps * 32;  // 320
constexpr int kMaxUnits = 9;                   // ceil(340*8 / 320)
constexpr int kEpiWarps = 8;                   // warps 4..11: (warp % 4) = TMEM lane quarter, (warp-4)/4 = MMA tile
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kMaxGnC = 512;
// GroupNorm statistics are accumulated as 64-bit fixed point (2^-24 resolution): integer atomics
// are associative, so the sums do not depend on the order in which CTAs finish.
constexpr double kStatScale = 16777216.0;
// Sums of squares reach 2 H W x^2 per channel pair and image; at 2^-24 they would wrap 63 bits once the activation rms
// approaches 1e3 at 512^2 (possible in the bf16 mode with a trained network).  Their scale is therefore a power of two
// chosen per tensor from its spatial size so that an rms of 65504 — the largest value the fp16 mode can store — still
// fits: 2^12 at 512^2, 2^14 at 256^2, ... (at most 2^24).  Producer and consumer of a tensor get it from the host.
__host__ __device__ inline double stat_sq_scale(long long hw) {
  int lg = 0;
  while ((1LL << lg) < hw) ++lg;
  int e = 30 - lg;
  e = e < 4 ? 4 : (e > 24 ? 24 : e);
  return double(1LL << e);
}

template <int N>
struct ConvCfg {
  static constexpr int kAccStride = N < 32 ? 32 : N;        // TMEM columns per 128-row accumulator
  static constexpr int kAccCols = 2 * kAccStride;           // two MMA tiles per CTA tile
  static constexpr int kNumAcc = (2 * kAccCols <= 512) ? 2 : 1;
  static constexpr int kNumAccMax = 2;  // half tiles (one MMA tile per CTA tile) double-buffer N = 256 as well
  // N = 64: per-lane running GroupNorm sums live in TMEM columns [256, 384)
  static constexpr bool kStatsInTmem = (N == 64);
  static constexpr int kStatCol0 = kNumAcc * kAccCols;
  static constexpr int kTmemNeed = kNumAcc * kAccCols + (kStatsInTmem ? 2 * N : 0);
  static constexpr int kTmemCols =
      kTmemNeed <= 32 ? 32 : (kTmemNeed <= 64 ? 64 : (kTmemNeed <= 128 ? 128 : (kTmemNeed <= 256 ? 256 : 512)));
  // a B stage holds as many consecutive tap blobs of one chunk as fit (N=64: 4 taps, 128: 2, 256: 1)
  // CTA pairs stage half-width blobs, so a stage of the same size holds twice the taps.  Cutting the same memory into
  // twice as many stages of half the size (more loads in flight) was measured 1.7 % SLOWER over the UNet (A/B on one
  // box, profiles/r2/ab_bsplit.log): the MMA warp's weight waits are shared-memory bandwidth (the bulk copies' writes
  // queue behind the tensor core's operand reads), not L2 latency, and more stages only add barrier work.
  static constexpr int kBStageBytes = N < 32 ? 9 * N * 128 : (N == 64 ? 24576 : 32768);
  // N <= 128 layers are bounded by the producer/epilogue roles, not by weight streaming: give the
  // input patch a third stage (deeper decoupling of producers and MMA) and the weights two.
  // (Measured: four patch stages with four one-tap weight stages for N = 64 removes the a_full waits
  // of the GroupNorm + 1x1-residual layers but starves the MMA warp of weights: 101 -> 132 us.)
  static constexpr int kAStages = N >= 256 ? 2 : 3;
  static constexpr int kBStages = N >= 256 ? 3 : 2;
  // N = 64 layers that mix a GroupNorm 3x3 chunk with 1x1-residual chunks split the patch memory into
  // two rings (ConvLayer::nG / nR): two full stages for the 3x3 chunks and two 32 KB stages for the dense
  // centre boxes.  In a single ring of three the 3x3 chunk of the next tile could only be requested two
  // (short) chunks before it is needed, which exposed its whole load + normalise latency every tile.
  static constexpr int kRStageBytes = kTileH * kTileW * 128;  // 32,768
  static constexpr int kASlots = N == 64 ? 4 : kAStages;       // mbarrier sets
  static constexpr int kABytes =
      N == 64 ? (2 * kAStageBytes + 2 * kRStageBytes > 3 * kAStageBytes ? 2 * kAStageBytes + 2 * kRStageBytes
                                                                        : 3 * kAStageBytes)
              : kAStages * kAStageBytes;
  static constexpr int kNcb = N < 32 ? 1 : N / 32;
  static constexpr int kRow = N < 32 ? 32 : N;  // floats per epilogue-warp statistics row
  // shared memory carve-up (bytes)
  static constexpr int kOffA = 0;
  static constexpr int kOffB = kOffA + kABytes;
  static constexpr int kOffTable = kOffB + kBStages * kBStageBytes;
  static constexpr int kOffBias = kOffTable + kMaxGnC * 8;
  static constexpr int kOffTstat = kOffBias + 256 * 4;
  static constexpr int kOffBar = kOffTstat + kEpiWarps * kRow * 4;  // one row of pair sums per epilogue warp
  // (+ the pair-mode relay barriers: the peer CTA's a_full / b_full / acc_empty as seen by the leader's MMA warp)
  static constexpr int kNumBar = 3 * kASlots + 2 * kBStages + 2 * kNumAccMax + (kASlots + kBStages + kNumAccMax);
  static constexpr int kOffTmem = kOffBar + kNumBar * 8;
  // per-epilogue-warp 2 KB staging block for the TMA store of 32 px x 32 ch (64B-swizzled)
  static constexpr int kOffStage = ((kOffTmem + 16 + 1023) / 1024) * 1024;
  // (N = 256: + 7 staging blocks of the second epilogue team, whose eighth block is the unused GroupNorm table)
  static constexpr int kSmemBytes = kOffStage + (N < 32 ? 0 : kEpiWarps * 2048) + (N >= 256 ? 7 * 2048 : 0);
  static_assert(kSmemBytes <= 232448, "exceeds the 227 KB of dynamic shared memory per CTA");
};

template <typename T>
struct Cvt;
template <>
struct Cvt<__half> {
  static constexpr int kFmt = 0;
  __device__ static __forceinline__ float2 unpack(uint32_t u) {
    return __half22float2(*reinterpret_cast<const __half2*>(&u));
  }
  __device__ static __forceinline__ uint32_t pack(float a, float b) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
  // activation store: saturate to +-65504 instead of producing inf (an inf becomes NaN in the next GroupNorm and
  // silently corrupts the image); the epilogue also raises the context's overflow flag, see kOverflowCheck
  __device__ static __forceinline__ uint32_t pack_store(float a, float b) {
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
  }
};
template <>
struct Cvt<__nv_bfloat16> {
  static constexpr int kFmt = 1;
  __device__ static __forceinline__ float2 unpack(uint32_t u) {
    return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u));
  }
  __device__ static __forceinline__ uint32_t pack(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
  __device__ static __forceinline__ uint32_t pack_store(float a, float b) { return pack(a, b); }  // fp32 exponent range
};

// swish(x*2sc + 2sh) for a packed pair, with sc/sh pre-halved: h = x*sc + sh; h*tanh(h) + h
__device__ __forceinline__ uint32_t swish_h2(uint32_t x, uint32_t sc, uint32_t sh) {
  uint32_t h, t, o;
  asm("fma.rn.f16x2 %0, %1, %2, %3;" : "=r"(h) : "r"(x), "r"(sc), "r"(sh));
  asm("tanh.approx.f16x2 %0, %1;" : "=r"(t) : "r"(h));
  asm("fma.rn.f16x2 %0, %1, %2, %1;" : "=r"(o) : "r"(h), "r"(t));
  return o;
}

// Operand format of a GroupNorm chunk.  fp16 mode: fp16.  bf16 mode: ALSO fp16 — activations are stored as bf16 (the
// un-normalised residual stream of a trained network may exceed the fp16 range), but what a GroupNorm chunk feeds the
// tensor core is swish(GroupNorm(x)), bounded by construction, so it is rounded to fp16 (11-bit significand instead of
// 8) and multiplied with fp16 weights; raw chunks (1x1 residual conv, up / down-sampling convs, stem) stay bf16 x bf16.
// tcgen05 kind::f16 takes the operand format per instruction.  This is what brings the bf16 mode inside the 1e-2
// per-step tolerance (SURVEY F10: bf16 operand rounding alone costs 0.9e-2).
template <typename T>
using GnOperand = __half;

// GroupNorm scale/shift + Swish on 8 packed 16-bit activations; the result is packed as GnOperand<T> (fp16).
// fp16 storage: packed fp16 throughout (hsc/hsh hold scale/2, shift/2): swish(y) = h tanh(h) + h, h = y/2.
// bf16 storage: the affine part in fp32 (sc/sh hold scale/2, shift/2; the input may be far outside the fp16 range),
//   then the same packed-half tanh form.
template <typename T>
__device__ __forceinline__ uint4 gn_swish_unit(uint4 o, const uint4& hsc, const uint4& hsh, const float (&sc)[8],
                                               const float (&sh)[8]) {
  if constexpr (Cvt<T>::kFmt == 0) {
    o.x = swish_h2(o.x, hsc.x, hsh.x);
    o.y = swish_h2(o.y, hsc.y, hsh.y);
    o.z = swish_h2(o.z, hsc.z, hsh.z);
    o.w = swish_h2(o.w, hsc.w, hsh.w);
    return o;
  } else {
    const uint32_t w4[4] = {o.x, o.y, o.z, o.w};
    uint32_t r4[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f = Cvt<T>::unpack(w4[e]);
      const float ya = fmaf(f.x, sc[2 * e], sh[2 * e]), yb = fmaf(f.y, sc[2 * e + 1], sh[2 * e + 1]);
      const uint32_t h = Cvt<__half>::pack(ya, yb);  // = y/2 (pre-halved table)
      uint32_t t;
      asm("tanh.approx.f16x2 %0, %1;" : "=r"(t) : "r"(h));
      asm("fma.rn.f16x2 %0, %1, %2, %1;" : "=r"(r4[e]) : "r"(h), "r"(t));
    }
    return make_uint4(r4[0], r4[1], r4[2], r4[3]);
  }
}

// GroupNorm scale/shift only (the SelfAttention norm of the SR3 baseline has no activation,
// ddpm_modules/unet.py:105,115): y = x*sc + sh; the tables hold sc/2, sh/2, so y = h + h.
template <typename T>
__device__ __forceinline__ uint4 gn_affine_unit(uint4 o, const uint4& hsc, const uint4& hsh, const float (&sc)[8],
                                                const float (&sh)[8]) {
  if constexpr (Cvt<T>::kFmt == 0) {
    const uint32_t w4[4] = {o.x, o.y, o.z, o.w}, s4[4] = {hsc.x, hsc.y, hsc.z, hsc.w}, b4[4] = {hsh.x, hsh.y, hsh.z, hsh.w};
    uint32_t r4[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      uint32_t h;
      asm("fma.rn.f16x2 %0, %1, %2, %3;" : "=r"(h) : "r"(w4[e]), "r"(s4[e]), "r"(b4[e]));
      asm("add.rn.f16x2 %0, %1, %1;" : "=r"(r4[e]) : "r"(h));
    }
    return make_uint4(r4[0], r4[1], r4[2], r4[3]);
  }
  const uint32_t w4[4] = {o.x, o.y, o.z, o.w};
  uint32_t r4[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float2 f = Cvt<T>::unpack(w4[e]);
    r4[e] = Cvt<GnOperand<T>>::pack(2.0f * fmaf(f.x, sc[2 * e], sh[2 * e]), 2.0f * fmaf(f.y, sc[2 * e + 1], sh[2 * e + 1]));
  }
  return make_uint4(r4[0], r4[1], r4[2], r4[3]);
}

// true in exactly one lane of a fully converged warp (elect.sync keeps the uniform datapath usable)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void named_bar_arrive(int id, int nthreads) {  // (the waiters call named_bar_sync)
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// 16-byte read-only global load, zero when !pred (no branch)
__device__ __forceinline__ uint4 ldg16_pred(const void* p, bool pred) {
  uint4 v;
  asm volatile(
      "{\n\t.reg .pred q;\n\t"
      "setp.ne.b32 q, %5, 0;\n\t"
      "mov.u32 %0, 0;\n\tmov.u32 %1, 0;\n\tmov.u32 %2, 0;\n\tmov.u32 %3, 0;\n\t"
      "@q ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];\n\t}"
      : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
      : "l"(p), "r"(int(pred)));
  return v;
}

// Transposing warp reduction: sum v[j] over the 32 lanes for all j at once.
// Generalisation to NV = 32, 16, 8 or 4 values per lane: lane l returns the 32-lane total of
// v[l >> (5 - log2 NV)] (replicated over 32/NV consecutive lanes).
template <int NV, int OFF, int NH>
struct TransposeReduceStep {
  __device__ static __forceinline__ void run(float (&v)[NV], int lane) {
    if constexpr (NH >= 1) {
      const bool up = (lane & OFF) != 0;
#pragma unroll
      for (int j = 0; j < NH; ++j) {
        const float keep = up ? v[j + NH] : v[j];
        const float send = up ? v[j] : v[j + NH];
        v[j] = keep + __shfl_xor_sync(0xffffffffu, send, OFF);
      }
    } else {
      v[0] += __shfl_xor_sync(0xffffffffu, v[0], OFF);
    }
    if constexpr (OFF > 1) TransposeReduceStep<NV, OFF / 2, NH / 2>::run(v, lane);
  }
};
template <int NV>
__device__ __forceinline__ float warp_transpose_reduce(float (&v)[NV], int lane) {
  TransposeReduceStep<NV, 16, NV / 2>::run(v, lane);
  return v[0];
}

// Optional role-level cycle accounting (tools/ only; compiled in with -DFDSR_PROFILE).
constexpr int kProfRoles = 5;  // 8 slots each per CTA: MMA, epilogue, producers, timeline, anchor
#ifdef FDSR_PROFILE
#define PROF_DECL long long pt_ = clock64(), pacc_[8] = {0, 0, 0, 0, 0, 0, 0, 0}
#define PROF_MARK(slot)              \
  do {                               \
    const long long n_ = clock64();  \
    pacc_[slot] += n_ - pt_;         \
    pt_ = n_;                        \
  } while (0)
#define PROF_FLUSH(role)                                                                  \
  do {                                                                                    \
    if (L.prof != nullptr)                                                                \
      for (int k_ = 0; k_ < 8; ++k_) L.prof[(size_t(blockIdx.x) * kProfRoles + (role)) * 8 + k_] = pacc_[k_]; \
  } while (0)
// timeline of one CTA (role 3): cycles since kernel entry at which an event FIRST happened (slot written once);
// role 4 anchors it: {SM id, the SM's clock64 at kernel entry, %globaltimer at entry} — consecutive launches on the
// same SM share the clock, which gives the idle time of the tensor pipe between two layers inside a running sampler
#define PROF_T0                                                                 \
  const long long pt0_ = clock64();                                             \
  if (threadIdx.x == 0 && L.prof != nullptr) {                                  \
    unsigned sm_;                                                               \
    long long gt_;                                                              \
    asm volatile("mov.u32 %0, %%smid;" : "=r"(sm_));                            \
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt_));                     \
    long long* p_ = L.prof + (size_t(blockIdx.x) * kProfRoles + 4) * 8;         \
    p_[0] = sm_;                                                                \
    p_[1] = pt0_;                                                               \
    p_[2] = gt_;                                                                \
  }
#define PROF_TS(slot)                                                                      \
  do {                                                                                     \
    if (L.prof != nullptr) L.prof[(size_t(blockIdx.x) * kProfRoles + 3) * 8 + (slot)] = clock64() - pt0_; \
  } while (0)
#define PROF_TS4(slot) /* anchor-row extras: 3 = accumulator of the CTA's last tile complete (tensor pipe drained) */ \
  do {                                                                                     \
    if (L.prof != nullptr) L.prof[(size_t(blockIdx.x) * kProfRoles + 4) * 8 + (slot)] = clock64() - pt0_; \
  } while (0)
#define PROF_PARAM , const long long pt0_  // (the role functions' timeline origin)
#define PROF_ARG , pt0_
#else
#define PROF_DECL
#define PROF_MARK(slot)
#define PROF_FLUSH(role)
#define PROF_T0
#define PROF_TS(slot)
#define PROF_TS4(slot)
#define PROF_PARAM
#define PROF_ARG
#endif

// kPair: CTA-pair form.  The kernel runs as clusters of two CTAs (one per SM of a TPC) and every MMA is a
//   tcgen05.mma.cta_group::2 of M = 256 rows: each CTA still owns a whole 32x8-pixel tile (its own input patch,
//   producers, TMEM accumulators and epilogue) but stages only HALF of the weight columns — CTA r supplies columns
//   [N/2 r, N/2 r + N/2) of B and the hardware exchanges the halves between the two SMs.  That halves both the weight
//   bytes written into shared memory per tile and the B bytes the tensor core reads per MMA: this kernel is bound by the
//   128 B/cycle of shared-memory bandwidth (an M128 x N64 x K16 MMA reads 4 KB of A + 2 KB of B for 32 cycles of math;
//   as a pair 4 KB + 1 KB).  The two tiles of a pair are x-neighbours (tile 2k + r), so they share the virtual image /
//   phase and therefore the weights.  Only the leader's warp 0 issues MMAs; the peer's warp 0 walks the same sequence
//   and forwards "my patch stage / weight half / accumulator is ready" to relay barriers in the leader's shared memory;
//   completions are multicast to both CTAs by tcgen05.commit.cta_group::2.
template <bool kPair>
constexpr int kTileStep = kPair ? 2 : 1;  // a CTA of a pair walks every second tile

// The order in which a CTA visits its tiles.  Every role walks it, and all must agree which tile a patch stage, a weight
// stage or an accumulator holds.  Tile t of the layer's order is tile (ty, tx) of virtual image b (phase layers:
// b = image * 4 + phase).  Only the constructor divides.  The tile grid is read from the layer (a constant-bank operand)
// at each step rather than copied into registers: the producer and epilogue roles already spill at 96 registers.
struct TileWalk {
  int b, ty, tx, step;
  const ConvLayer* L;
  TileWalk() = default;
  __device__ __forceinline__ TileWalk(int t, const ConvLayer& layer, int step_) : step(step_), L(&layer) {
    b = t / (L->tiles_x * L->tiles_y);
    ty = (t - b * L->tiles_x * L->tiles_y) / L->tiles_x;
    tx = t - (b * L->tiles_y + ty) * L->tiles_x;
  }
  __device__ __forceinline__ void advance() {
    if ((tx += step) >= L->tiles_x) {
      tx -= L->tiles_x;
      if (++ty == L->tiles_y) { ty = 0; ++b; }
    }
  }
  __device__ __forceinline__ TileWalk peek_next() const { TileWalk n = *this; n.advance(); return n; }
};

// Cursor over a ring of n stages whose barriers flip phase once per lap.
struct StageRing {
  int slot = 0, phase = 0;
  __device__ __forceinline__ void advance(int n) { if (++slot == n) { slot = 0; phase ^= 1; } }
};

// mbarrier addresses (8 bytes each from ConvCfg::kOffBar; kNumBar counts them).  raw_full: TMA-fed layers, the raw patch
// of the stage has landed.  pa_full / pb_full / pacc_empty: pair-mode relay barriers (used in the leader CTA only;
// arrivals come from the peer's warp 0).
template <int N>
struct ConvBars {
  using Cfg = ConvCfg<N>;
  static constexpr int kA = Cfg::kASlots, kB = 2 * kA, kAcc = kB + 2 * Cfg::kBStages, kRaw = kAcc + 2 * Cfg::kNumAccMax,
                       kRelay = kRaw + kA;
  uint32_t bar0;
  __device__ __forceinline__ uint32_t a_full(int s) const { return bar0 + 8u * s; }
  __device__ __forceinline__ uint32_t a_empty(int s) const { return bar0 + 8u * (kA + s); }
  __device__ __forceinline__ uint32_t b_full(int s) const { return bar0 + 8u * (kB + s); }
  __device__ __forceinline__ uint32_t b_empty(int s) const { return bar0 + 8u * (kB + Cfg::kBStages + s); }
  __device__ __forceinline__ uint32_t acc_full(int s) const { return bar0 + 8u * (kAcc + s); }
  __device__ __forceinline__ uint32_t acc_empty(int s) const { return bar0 + 8u * (kAcc + Cfg::kNumAccMax + s); }
  __device__ __forceinline__ uint32_t raw_full(int s) const { return bar0 + 8u * (kRaw + s); }
  __device__ __forceinline__ uint32_t pa_full(int s) const { return bar0 + 8u * (kRelay + s); }
  __device__ __forceinline__ uint32_t pb_full(int s) const { return bar0 + 8u * (kRelay + kA + s); }
  __device__ __forceinline__ uint32_t pacc_empty(int s) const { return bar0 + 8u * (kRelay + kA + Cfg::kBStages + s); }
};

// The CTA's tiles and the geometry every role derives from the layer (computed once in the kernel body).
template <int N>
struct ConvSched {
  int tile_begin, tile_end;  // the CTA's tiles (pair mode: tile pairs)
  int tile_first;            // index of the CTA's first tile in the layer's tile order
  TileWalk first;            // ... and the walk from it (the epilogue's tail helpers start elsewhere)
  uint32_t crank;            // 0 = leader of a pair (issues the MMAs) or single CTA, 1 = peer
  int TH, nacc, taps_per_stage, n_off, nG, nR;  // tile rows; accumulator stages; split-N: first output channel
  bool two_mt;                                  // two 128-row MMA tiles per CTA tile
  uint32_t acc_cols, blob, gblob;  // TMEM columns per accumulator; bytes of a tap's weight blob: staged / in global memory
  // patch rings: slots [0, nG) are full stages (ring 0), slots [nG, nG + nR) 32 KB centre-box stages (ring 1)
  __device__ __forceinline__ uint32_t slot_off(int slot) const {
    return uint32_t(slot < nG ? slot * kAStageBytes : nG * kAStageBytes + (slot - nG) * ConvCfg<N>::kRStageBytes);
  }
};

// =========================================================== MMA issuer (whole warp converged, tcgen05 instructions
// issued by the elected lane)
template <int N, typename T, bool kPair>
__device__ __forceinline__ void mma_role(const ConvLayer& L, const ConvSched<N>& S, const ConvBars<N>& bars,
                                         uint32_t tmem, uint8_t* smem PROF_PARAM) {
  using Cfg = ConvCfg<N>;
  constexpr int NB = kPair ? N / 2 : N;  // weight columns this CTA stages
  const int lane = threadIdx.x & 31;
  const uint32_t sA = smem_u32(smem + Cfg::kOffA), sB = smem_u32(smem + Cfg::kOffB);
  const uint32_t idesc_raw = make_idesc_f16(kPair ? 256 : 128, N, Cvt<T>::kFmt);
  const uint32_t idesc_gn = make_idesc_f16(kPair ? 256 : 128, N, Cvt<GnOperand<T>>::kFmt);  // (see GnOperand)
  const bool leader = S.crank == 0;  // (pair mode: the peer's warp 0 only forwards its barriers to the leader)
  // descriptor = hi:lo; hi is constant, lo = (LBO>>4)<<16 | (addr>>4), advanced by plain adds
  // A operand: no-swizzle channel-group planes (SBO = 10 positions x 16 B, LBO = plane) when the
  // producers gather it, 128B-swizzled pixel-major rows (SBO = 10 positions x 128 B, layout type 2)
  // when TMA delivers it; the hardware swizzle is a function of the absolute shared-memory address
  // (tools/probe_umma.cu layouts 3/4), so a tap is still just a shifted start address.
  const bool sw = L.a_tma == 1;
  const uint32_t a_hi_full = sw ? (((kPatchW * 128) >> 4) | (1u << 14) | (2u << 29)) : (((kPatchW * 16) >> 4) | (1u << 14));
  const uint32_t a_hi_cen = ((kTileW * 128) >> 4) | (1u << 14) | (2u << 29);
  const uint32_t b_hi = (128u >> 4) | (1u << 14);
  // (inside a cluster, shared-window addresses carry the CTA rank above bit 18: keep the 18-bit offset)
  const uint32_t plane16 = L.a_tma == 2 ? uint32_t(kPlaneBytesTma >> 4) : uint32_t(kPlaneBytes >> 4);
  const uint32_t a_lo0 = ((sw ? 1u : plane16) << 16) + ((sA & 0x3FFFFu) >> 4);
  const uint32_t kstep = sw ? 2u : 2u * plane16;  // 16-byte units between K = 16 slices
  const int pos_sh = sw ? 3 : 0;                    // patch position -> 16-byte units
  const uint32_t mt1_full = uint32_t(16 * kPatchW) << pos_sh;  // second 128-row MMA tile: 16 image rows down
  const uint32_t b_lo0 = (uint32_t((NB * 16) >> 4) << 16) + ((sB & 0x3FFFFu) >> 4);
  const int ksteps = L.ncg >> 1;
  StageRing ga, ra, bst, acc;  // patch ring 0, patch ring 1, weight stages, accumulators
  // Weight stages hold taps_per_stage consecutive taps of the CTA's whole tap stream (all chunks of a
  // tile, tile after tile), so a stage may end in the middle of a chunk and a chunk in the middle of a
  // stage: bq = taps of the current stage already consumed.
  int bq = 0;
  // phase layers (L.phases = 4): tiles run over virtual images bv = image * 4 + (py * 2 + px); the 2x2 taps of
  // phase (py, px) are the phase-0 taps shifted by (py, px) positions inside the low-resolution patch
  TileWalk walk = S.first;
  // Pair mode hand-shake.  A barrier the MMA warp waits for exists in both CTAs (each CTA's producers, loader and
  // epilogue only ever talk to their own); the peer's warp 0 waits for its local one and then arrives on the relay
  // barrier of the same stage in the leader's shared memory, which the leader waits for after its own.  The k-th use
  // of a stage completes phase k-1 of its relay barrier (also for acc_empty, whose first local wait falls through).
  auto pair_sync = [&](uint32_t relay_bar, uint32_t use_parity) {
    if constexpr (kPair) {
      if (leader) mbar_wait(relay_bar, use_parity);
      else if (lane == 0) mbar_arrive_remote(relay_bar, 0);
      __syncwarp();
    }
  };
  PROF_DECL;
  for (int tile = S.tile_begin; tile < S.tile_end; ++tile) {
    mbar_wait(bars.acc_empty(acc.slot), acc.phase ^ 1);
    pair_sync(bars.pacc_empty(acc.slot), acc.phase);
    PROF_MARK(0);
    tc_fence_after();
    const uint32_t d0 = tmem + acc.slot * S.acc_cols;
    const uint32_t phoff = L.phases > 1 ? uint32_t(((walk.b >> 1) & 1) * kPatchW + (walk.b & 1)) << pos_sh : 0u;
    walk.advance();
    for (int c = 0; c < L.nchunks; ++c) {
      const ConvChunk& ck = L.chunk[c];
      const int ntaps = ck.ntaps;
      const bool r1 = ck.ring != 0;
      const int as = r1 ? S.nG + ra.slot : ga.slot, aph = r1 ? ra.phase : ga.phase;
      const uint32_t idesc = ck.gn != 0 ? idesc_gn : idesc_raw;
      mbar_wait(bars.a_full(as), aph);
      pair_sync(bars.pa_full(as), aph);
      PROF_MARK(1);
      const uint32_t a_stage = a_lo0 + (S.slot_off(as) >> 4);
      // centre-box chunk (raw single-tap chunk of a TMA-fed layer): dense 32x8 positions, no halo
      const bool cen = ck.center != 0;
      const uint32_t a_hi = cen ? a_hi_cen : a_hi_full;
      const uint32_t mt1 = cen ? uint32_t(16 * kTileW) << 3 : mt1_full;
      for (int tp0 = 0; tp0 < ntaps;) {
        const int g = ntaps - tp0 < S.taps_per_stage - bq ? ntaps - tp0 : S.taps_per_stage - bq;
        if (bq == 0) {
          mbar_wait(bars.b_full(bst.slot), bst.phase);
          pair_sync(bars.pb_full(bst.slot), bst.phase);
        }
        PROF_MARK(2);
        tc_fence_after();
        const bool stage_done = bq + g == S.taps_per_stage;
        if (leader && elect_one()) {
          if (tile == S.tile_begin && c == 0 && tp0 == 0) PROF_TS(4);  // first MMA issued
          uint32_t b_lo = b_lo0 + bst.slot * (Cfg::kBStageBytes >> 4) + bq * (S.blob >> 4);
          for (int tg = 0; tg < g; ++tg, b_lo += S.blob >> 4) {
            const uint32_t a_lo = a_stage + (cen ? 0u : (uint32_t(ck.tap_pos[tp0 + tg]) << pos_sh) + phoff);
            const uint32_t accum0 = (c | tp0 | tg) == 0 ? 0u : 1u;
            auto issue = [&](int ks) {
              const uint64_t bd = (uint64_t(b_hi) << 32) | (b_lo + ks * 2 * NB);
              const uint64_t ad0 = (uint64_t(a_hi) << 32) | (a_lo + ks * kstep);
              const uint64_t ad1 = (uint64_t(a_hi) << 32) | (a_lo + ks * kstep + mt1);
              if constexpr (kPair) {
                umma_f16_pair(d0, ad0, bd, idesc, ks ? 1u : accum0);
                if (S.two_mt) umma_f16_pair(d0 + Cfg::kAccStride, ad1, bd, idesc, ks ? 1u : accum0);
              } else {
                umma_f16(d0, ad0, bd, idesc, ks ? 1u : accum0);
                if (S.two_mt) umma_f16(d0 + Cfg::kAccStride, ad1, bd, idesc, ks ? 1u : accum0);
              }
            };
            if (ksteps == 4) {
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) issue(ks);
            } else {
              for (int ks = 0; ks < ksteps; ++ks) issue(ks);
            }
          }
          auto commit = [&](uint32_t bar) {
            if constexpr (kPair) umma_commit_pair(bar);
            else umma_commit(bar);
          };
          if (stage_done) commit(bars.b_empty(bst.slot));  // (the last, partial stage of the CTA is never waited for)
          if (tp0 + g >= ntaps) commit(bars.a_empty(as));
          if (tp0 + g >= ntaps && c == L.nchunks - 1) {
            commit(bars.acc_full(acc.slot));
            if (tile + 1 == S.tile_end) PROF_TS(5);  // last MMA of the CTA issued
          }
        }
        __syncwarp();
        PROF_MARK(3);
        tp0 += g;
        bq += g;
        if (stage_done) {
          bq = 0;
          bst.advance(Cfg::kBStages);
        }
      }
      if (r1) ra.advance(S.nR);
      else ga.advance(S.nG);
    }
    acc.advance(S.nacc);
  }
  if (lane == 0) PROF_FLUSH(0);
}

// =========================================================== loader: weight stages (bulk copies of pre-packed tap
// blobs) and, for TMA-fed layers, the input patches (one tensor load per chunk).
// Two independent cursors polled in one loop: a patch is requested the moment its stage is
// released (up to kAStages chunks ahead of the MMA warp), a weight stage the moment it is free.
// GroupNorm chunks land on raw_full (the producer warps transform them in place and then arrive on
// a_full); raw chunks complete a_full directly, so the MMA warp starts as soon as the bytes are there.
template <int N, typename T, bool kPair>
__device__ __forceinline__ void loader_role(const ConvLayer& L, const ConvSched<N>& S, const ConvBars<N>& bars,
                                            uint8_t* smem) {
  using Cfg = ConvCfg<N>;
  const uint32_t sA = smem_u32(smem + Cfg::kOffA), sB = smem_u32(smem + Cfg::kOffB);
  const uint32_t patch_bytes = uint32_t((S.TH + 2) * kPatchW) * 128u, cen_bytes = uint32_t(S.TH) * kTileW * 128u;
  const bool tma_in = L.a_tma != 0;
  const int ncg = L.ncg, n_full = L.n_full;  // (read once: the bulk copies' memory clobber would force reloads per copy)
  // Patches are the previous layer's output: no patch request before griddepcontrol.wait.  The loader of a TMA-fed
  // layer waits for it before its first weight stage too, so that the first patch is requested first: a CTA only
  // becomes resident when the previous launch's CTA on this SM has exited, so the dependency resolves within a few
  // microseconds anyway, and 64 - 96 KB of weight stages queued ahead of the 43 KB patch on the SM's inbound link
  // would delay the longer chain (patch -> GroupNorm pass -> first MMA; the weights are only needed at the end of it).
  // Measured -0.6 % of a UNet step's op time, -1.6 % of the sampler at B = 16 (profiles/r2/ab_tail.log).
  if (tma_in) asm volatile("griddepcontrol.wait;" ::: "memory");
  const int total = (S.tile_end - S.tile_begin) * L.nchunks;
  // patch cursor
  int a_next = tma_in ? 0 : total, a_c = 0;
  StageRing a_ga, a_ra;
  TileWalk a_walk = S.first;
  // weight cursor: stage-loads of taps_per_stage taps over the periodic tap stream (period = taps per tile;
  // all chunks of a layer have equally sized tap blobs, packed back to back in chunk order)
  int taps_tile = 0;
  for (int c = 0; c < L.nchunks; ++c) taps_tile += L.chunk[c].ntaps;
  const int total_taps = (S.tile_end - S.tile_begin) * taps_tile;
  int b_q = 0, b_qq = 0;  // next tap overall / inside its tile
  StageRing bst;
  // (pair mode: the weights are packed as two half-width copies of the single-CTA layout, half r for CTA r)
  const uint8_t* const w0 = L.weights + (kPair ? size_t(S.crank) * size_t(L.w_half) : size_t(S.n_off) * 16);
  // phase layers: the weights of phase p follow those of phase p-1 (taps_tile blobs each); w_walk.b = virtual image of
  // the tile that tap b_q belongs to
  const int phsh = L.phases > 1 ? 2 : 0;
  const size_t ph_stride = L.phases > 1 ? size_t(taps_tile) * (kPair ? S.blob : S.gblob) : 0;
  TileWalk w_walk = S.first;
  while (a_next < total || b_q < total_taps) {
    bool progress = false;
    if (a_next < total) {
      const bool a_r1 = L.chunk[a_c].ring != 0;
      const int a_as = a_r1 ? S.nG + a_ra.slot : a_ga.slot;
      const uint32_t ok = mbar_test(bars.a_empty(a_as), (a_r1 ? a_ra.phase : a_ga.phase) ^ 1) ? 1u : 0u;
      if (__shfl_sync(0xffffffffu, ok, 0)) {
        if (elect_one()) {
          const ConvChunk& ak = L.chunk[a_c];
          const uint32_t dst = sA + S.slot_off(a_as);
          const int a_b = a_walk.b, a_ty = a_walk.ty, a_tx = a_walk.tx;
          if (L.a_tma == 2) {
            // 16-channel stem input: two 8-channel planes (box 8 ch x 10 x 34, no swizzle) land as the
            // [channel group][position][8 ch] patch the gathered layers use; nothing for the producer warps to do
            const uint32_t bar = bars.a_full(a_as);
            mbar_arrive_cnt(bar, kProdWarps - 1);
            mbar_arrive_expect_tx(bar, 2 * kPatchPos * 16);
            tma_load_4d(&L.in_map[ak.src], dst, bar, ak.c0, a_tx * kTileW - 1, a_ty * kTileH - 1, a_b);
            tma_load_4d(&L.in_map[ak.src], dst + kPlaneBytesTma, bar, ak.c0 + 8, a_tx * kTileW - 1, a_ty * kTileH - 1, a_b);
          } else if (ak.gn != 0) {
            mbar_arrive_expect_tx(bars.raw_full(a_as), patch_bytes);
            tma_load_4d(&L.in_map[ak.src], dst, bars.raw_full(a_as), ak.c0, a_tx * kTileW - 1, a_ty * S.TH - 1, a_b >> phsh);
          } else {
            const uint32_t bar = bars.a_full(a_as);
            mbar_arrive_cnt(bar, kProdWarps - 1);  // stands in for the producer warps
            if (L.mode == kModeS2D) {  // parity plane (pa, pb) of the stride-2 conv's input: every second pixel
              mbar_arrive_expect_tx(bar, patch_bytes);
              tma_load_4d(&L.in_map_c[ak.src], dst, bar, ak.c0, 2 * (a_tx * kTileW - 1) + (ak.parity & 1),
                          2 * (a_ty * S.TH - 1) + (ak.parity >> 1), a_b);
            } else if (ak.center != 0) {
              mbar_arrive_expect_tx(bar, cen_bytes);
              tma_load_4d(&L.in_map_c[ak.src], dst, bar, ak.c0, a_tx * kTileW, a_ty * S.TH, a_b >> phsh);
            } else {
              mbar_arrive_expect_tx(bar, patch_bytes);
              tma_load_4d(&L.in_map[ak.src], dst, bar, ak.c0, a_tx * kTileW - 1, a_ty * S.TH - 1, a_b >> phsh);
            }
          }
        }
        __syncwarp();
        ++a_next;
        if (a_r1) a_ra.advance(S.nR);
        else a_ga.advance(S.nG);
        if (++a_c == L.nchunks) {
          a_c = 0;
          a_walk.advance();
        }
        progress = true;
      }
    }
    if (b_q < total_taps) {
      const uint32_t ok = mbar_test(bars.b_empty(bst.slot), bst.phase ^ 1) ? 1u : 0u;
      if (__shfl_sync(0xffffffffu, ok, 0)) {
        const int g = total_taps - b_q < S.taps_per_stage ? total_taps - b_q : S.taps_per_stage;
        if (elect_one()) {
          mbar_arrive_expect_tx(bars.b_full(bst.slot), uint32_t(g) * S.blob);
          const uint32_t dst0 = sB + bst.slot * Cfg::kBStageBytes;
          if (L.nsplit == 1) {
            // contiguous runs up to the end of each tile's taps (the next tile may belong to another phase)
            int rem = g, qq = b_qq;
            TileWalk t = w_walk;
            uint32_t dst = dst0;
            while (rem > 0) {
              const int n = rem < taps_tile - qq ? rem : taps_tile - qq;
              bulk_g2s(dst, w0 + size_t(t.b & 3) * ph_stride + size_t(qq) * S.blob, uint32_t(n) * S.blob, bars.b_full(bst.slot));
              dst += uint32_t(n) * S.blob;
              rem -= n;
              qq += n;
              if (qq == taps_tile) {
                qq = 0;
                t.advance();
              }
            }
          } else {
            int qq = b_qq;
            TileWalk t = w_walk;
            for (int tg = 0; tg < g; ++tg) {
              const uint8_t* wt = w0 + size_t(t.b & 3) * ph_stride + size_t(qq) * S.gblob;
              const uint32_t dst = dst0 + uint32_t(tg) * S.blob;
              // this CTA's N of the n_full columns: one contiguous run per channel group
              for (int cgi = 0; cgi < ncg; ++cgi)
                bulk_g2s(dst + uint32_t(cgi) * N * 16, wt + size_t(cgi) * n_full * 16, N * 16, bars.b_full(bst.slot));
              if (++qq == taps_tile) {
                qq = 0;
                t.advance();
              }
            }
          }
        }
        __syncwarp();
        bst.advance(Cfg::kBStages);
        b_q += g;
        for (b_qq += g; b_qq >= taps_tile; b_qq -= taps_tile) w_walk.advance();
        progress = true;
      }
    }
    if (!progress) __nanosleep(32);
  }
}

// =========================================================== input producers (warps 2, 3, 12..19)
template <int N, typename T, bool kPair>
__device__ __forceinline__ void producer_role(const ConvLayer& L, const ConvSched<N>& S, const ConvBars<N>& bars,
                                              uint8_t* smem PROF_PARAM) {
  using Cfg = ConvCfg<N>;
  constexpr int kAStages = Cfg::kAStages;  // gathered layers: one ring of kAStages full stages
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int pw = warp < 4 ? warp - 2 : warp - 10;  // warps 2,3,12..19 -> 0..9
  const int pidx = pw * 32 + lane;                  // 0..319
  __builtin_assume(pidx >= 0 && pidx < kProdThreads);  // (known to the dispatch, not to this function: folds the unit masks)
  const int H = L.H, W = L.W, TH = S.TH;
  const int npos = (TH + 2) * kPatchW;  // patch positions (340 / 180)
  const uint32_t sA = smem_u32(smem + Cfg::kOffA);
  float2* table = reinterpret_cast<float2*>(smem + Cfg::kOffTable);
  __half* table_h = reinterpret_cast<__half*>(table);
  int cur_b = -1;
  TileWalk walk = S.first;
  PROF_DECL;

  // GroupNorm scale/shift table of sample `bb` (virtual concat of the GroupNorm sources).
  // Everything that does not depend on the previous launch — gamma / beta of this thread's two channels, the pair
  // range of their groups, the reciprocals — is fetched BEFORE griddepcontrol.wait; afterwards a table costs one
  // round of independent statistics loads (every thread sums the <= 8 channel pairs of its own group straight from
  // L2: no staging, no cross-thread hand-off), three fp64 operations, an rsqrt and one barrier.  This sits on the
  // critical path of every launch (statistics -> table -> first normalised patch -> first MMA).
  const int cpg = L.gn_C > 0 ? L.gn_C / L.gn_groups : 2, ppg = cpg >> 1, p0 = L.src[0].C >> 1;
  float ga[2] = {0.f, 0.f}, be[2] = {0.f, 0.f};
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const int c = pidx + j * kProdThreads;
    if (c < L.gn_C) {
      ga[j] = L.gamma[c];
      be[j] = L.beta[c];
    }
  }
  const double inv_sum = L.gn_inv_sum, inv_sq = L.gn_inv_sq;  // 1 / (fixed-point scale * elements per group), host-side
  bool table_valid = false;
#ifdef FDSR_PROFILE
  uint4 probe_ = make_uint4(0u, 0u, 0u, 0u);  // (timeline only) one plain 16-byte load of the first patch's first pixel
#endif
  auto build_table = [&](int bb) {
    const bool first_table = !table_valid;
    (void)first_table;
    if (table_valid) named_bar_sync(1, kProdThreads);  // everyone is done reading the previous table
    table_valid = true;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int c = pidx + j * kProdThreads;
      if (c < L.gn_C) {
        const int pv0 = (c / cpg) * ppg;
        long long Si = 0, Qi = 0;
#pragma unroll 8
        for (int k = 0; k < ppg; ++k) {
          const int pv = pv0 + k;
          const int si = pv < p0 ? 0 : 1;
          const int pl = pv < p0 ? pv : pv - p0;
          const longlong2 st = __ldg(reinterpret_cast<const longlong2*>(
              reinterpret_cast<const long long*>(L.src[si].stats) + (size_t(bb) * (L.src[si].C >> 1) + pl) * 2));
          Si += st.x;
          Qi += st.y;
        }
#ifdef FDSR_PROFILE
        if (pidx == 0 && j == 0 && first_table) {
          long long z_;
          asm volatile("and.b64 %0, %1, 0;" : "=l"(z_) : "l"(Si + Qi));  // (the statistics have arrived)
          if (z_ == 0) PROF_TS4(5);
          unsigned z2_;
          asm volatile("and.b32 %0, %1, 0;" : "=r"(z2_) : "r"(probe_.x ^ probe_.w));  // (... and the probe load)
          if (z2_ == 0) PROF_TS4(7);
        }
#endif
        const double mean = double(Si) * inv_sum;
        double var = double(Qi) * inv_sq - mean * mean;
        var = var > 0.0 ? var : 0.0;
        const float rstd = rsqrtf(float(var) + L.gn_eps);
        const float sc = ga[j] * rstd;
        const float sh = be[j] - float(mean) * sc;
        // half-scaled so that swish(y) = h*tanh(h) + h with h = y/2
        if constexpr (Cvt<T>::kFmt == 0) {
          table_h[c] = __float2half_rn(0.5f * sc);
          table_h[kMaxGnC + c] = __float2half_rn(0.5f * sh);
        } else {  // bf16 storage: fp32 affine, then the packed-half tanh form
          table[c] = make_float2(0.5f * sc, 0.5f * sh);
        }
      }
    }
    if (pidx == 0 && first_table) PROF_TS4(6);  // table entries of this thread written
    named_bar_sync(1, kProdThreads);
  };
  // (a dry run of build_table on stale statistics before the wait, to warm its code path, measured 0.4 % slower)
  asm volatile("griddepcontrol.wait;" ::: "memory");
  if (pidx == 0) PROF_TS4(4);  // (producers) previous launch complete
#ifdef FDSR_PROFILE
  if (pidx == 0 && L.a_tma == 1 && L.gn_C > 0 && L.phases == 1 && S.tile_end > S.tile_begin) {
    const ConvSrc& s0 = L.src[L.chunk[0].src];
    const int yy = walk.ty * TH - 1 < 0 ? 0 : walk.ty * TH - 1, xx = walk.tx * kTileW - 1 < 0 ? 0 : walk.tx * kTileW - 1;
    probe_ = ldg16_pred(reinterpret_cast<const uint8_t*>(s0.ptr) +
                            ((size_t(walk.b) * s0.H + yy) * s0.W + xx) * size_t(s0.C) * 2 + size_t(L.chunk[0].c0) * 2, true);
  }
#endif
  if (L.a_tma != 0) {
    // ----------------------------------------------------------------- TMA-fed layers: the loader warp's
    // tensor loads land the raw 128B-swizzled patch in the stage (out-of-image positions zero);
    // these warps apply GroupNorm + Swish in place and hand the stage to the MMA warp.  The thread
    // owns 16-byte slot (pidx & 7) of positions (pidx >> 3) + 40 i: byte pidx*16 + i*5120 of the stage
    // (conflict-free: a warp covers 512 contiguous bytes).  40 positions are 5 swizzle periods, so the
    // slot's logical channel group depends only on the stage
    // (stage s starts 341 s = 5 s mod 8 rows into the swizzle period)
    const int pos0 = pidx >> 3;
    const int py0 = pos0 / kPatchW, px0 = pos0 - py0 * kPatchW;  // position of unit i: (py0 + 4 i, px0)
    uint32_t smask = 0u;  // unit i = position pos0 + 40 i exists in the (TH + 2) x 10 patch
#pragma unroll
    for (int i = 0; i < kMaxUnits; ++i) smask |= (pos0 + 40 * i < npos) ? (1u << i) : 0u;
    // ring 0 only (ring-1 chunks are raw).  raw_full(s) completes only for the GroupNorm chunks that use slot s, not on
    // every lap of the ring (raw ring-0 chunks complete a_full directly), so its parity is kept per slot: bit s
    StageRing ring;
    uint32_t rph = 0u;
    for (int tile = S.tile_begin; tile < S.tile_end; ++tile) {
      // units inside the image (padding must stay zero: swish(GN(0)) != 0)
      const int y0 = walk.ty * TH - 1 + py0, x0 = walk.tx * kTileW - 1 + px0;
      uint32_t vmask = 0u;
      if (unsigned(x0) < unsigned(W)) {
#pragma unroll
        for (int i = 0; i < kMaxUnits; ++i) vmask |= unsigned(y0 + 4 * i) < unsigned(H) ? (1u << i) : 0u;
        vmask &= smask;
      }
      // (Tried and dropped — the first data of a launch arrives ~3 us after its dependency resolves, whatever asks for
      //  it: gathering the CTA's first patch with plain loads from these threads, holding the weight requests back until
      //  the first patch has landed, prefetching the tensor maps: none was faster; profiles/r2/ab_first_ldg.log,
      //  ab_hold.log, ab_tensormap_prefetch.log.  A plain 16-byte load issued at the dependency returns after 1.3 us.)
      if (L.gn_C > 0 && walk.b != cur_b) {
        cur_b = walk.b;
        build_table(walk.b);
        if (pidx == 0 && tile == S.tile_begin) PROF_TS(2);  // GroupNorm table of the first image built
      }
      PROF_MARK(0);
      for (int c = 0; c < L.nchunks; ++c) {
        const ConvChunk& ck = L.chunk[c];
        if (ck.gn == 0) {  // raw chunk: the tensor load completes a_full by itself
          if (ck.ring == 0) ring.advance(S.nG);
          continue;
        }
        const int as = ring.slot;
        mbar_wait(bars.raw_full(as), (rph >> as) & 1u);
        rph ^= 1u << as;
        if (pidx == 0 && tile == S.tile_begin && c == 0) PROF_TS(3);  // first patch landed
        PROF_MARK(1);
        const int cgs = (pidx & 7) ^ ((pos0 + 5 * as) & 7);
        float sc[8], sh[8];
        uint4 hsc = make_uint4(0u, 0u, 0u, 0u), hsh = hsc;
        if constexpr (Cvt<T>::kFmt == 0) {
          hsc = *reinterpret_cast<const uint4*>(table_h + ck.vc0 + cgs * 8);
          hsh = *reinterpret_cast<const uint4*>(table_h + kMaxGnC + ck.vc0 + cgs * 8);
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float2 e = table[ck.vc0 + cgs * 8 + j];
            sc[j] = e.x;
            sh[j] = e.y;
          }
        }
        const uint32_t a0 = sA + as * kAStageBytes + uint32_t(pidx) * 16;  // (GroupNorm chunks: ring 0)
        uint4 rv[kMaxUnits];
#pragma unroll
        for (int i = 0; i < kMaxUnits; ++i)
          if ((vmask >> i) & 1u) rv[i] = lds128(a0 + i * (40 * 128));
        if (ck.gn == 1) {
#pragma unroll
          for (int i = 0; i < kMaxUnits; ++i)
            if ((vmask >> i) & 1u) sts128(a0 + i * (40 * 128), gn_swish_unit<T>(rv[i], hsc, hsh, sc, sh));
        } else {  // GroupNorm without activation
#pragma unroll
          for (int i = 0; i < kMaxUnits; ++i)
            if ((vmask >> i) & 1u) sts128(a0 + i * (40 * 128), gn_affine_unit<T>(rv[i], hsc, hsh, sc, sh));
        }
        fence_proxy_async_smem();
        PROF_MARK(3);
        __syncwarp();
        if (lane == 0) mbar_arrive(bars.a_full(as));
        ring.advance(S.nG);
      }
      walk.advance();
    }
  } else {
    // ----------------------------------------------------------------- nearest-upsample convs in the nine-tap form
    // (64-channel raw chunks, no GroupNorm): predicated 16-byte global loads of the 2x-upsampled patch, 16-byte stores
    // into the no-swizzle [channel group][position][8 ch] patch
    const int cg = pidx & 7;
    // per-thread patch coordinates of the (up to) 9 16-byte units it fills: fixed for the launch
    uint32_t pcoord[kMaxUnits];  // py | px << 8
    uint32_t smask = 0u;         // bit i: unit i has a smem slot to fill
#pragma unroll
    for (int i = 0; i < kMaxUnits; ++i) {
      const int u = pidx + i * kProdThreads;
      const int pos = u >> 3;
      const int py = pos / kPatchW, px = pos - py * kPatchW;
      smask |= u < kPatchPos * 8 ? (1u << i) : 0u;
      pcoord[i] = uint32_t(py) | (uint32_t(px) << 8);
    }
    const int src_w = W >> 1;
    StageRing ring;
    for (int tile = S.tile_begin; tile < S.tile_end; ++tile) {
      const int y0 = walk.ty * kTileH - 1, x0 = walk.tx * kTileW - 1;
      // ---- source pixel offsets of this thread's patch positions; vmask bit i = inside the image
      int pixoff[kMaxUnits];
      uint32_t vmask = 0u;
#pragma unroll
      for (int i = 0; i < kMaxUnits; ++i) {
        const int y = y0 + int(pcoord[i] & 0xffu), x = x0 + int((pcoord[i] >> 8) & 0xffu);
        const bool ok = ((smask >> i) & 1u) != 0u && unsigned(y) < unsigned(H) && unsigned(x) < unsigned(W);
        const int off = (y >> 1) * src_w + (x >> 1);
        pixoff[i] = ok ? off : 0;
        vmask |= ok ? (1u << i) : 0u;
      }
      PROF_MARK(0);
      for (int c = 0; c < L.nchunks; ++c) {
        const ConvChunk& ck = L.chunk[c];
        const ConvSrc& s = L.src[ck.src];
        const int sC = s.C;
        const uint8_t* base = reinterpret_cast<const uint8_t*>(
            reinterpret_cast<const T*>(s.ptr) + size_t(walk.b) * s.H * s.W * sC + ck.c0 + cg * 8);
        const uint32_t pix_bytes = uint32_t(sC) * 2u;
        uint4 rv[kMaxUnits];
#pragma unroll
        for (int i = 0; i < kMaxUnits; ++i)
          rv[i] = ldg16_pred(base + uint32_t(pixoff[i]) * pix_bytes, ((vmask >> i) & 1u) != 0u);
        PROF_MARK(1);
        mbar_wait(bars.a_empty(ring.slot), ring.phase ^ 1);
        PROF_MARK(2);
        const uint32_t dst0 = sA + ring.slot * kAStageBytes + cg * kPlaneBytes + uint32_t(pidx >> 3) * 16;
#pragma unroll
        for (int i = 0; i < kMaxUnits; ++i)
          if ((smask >> i) & 1u) sts128(dst0 + uint32_t((i * kProdThreads) >> 3) * 16, rv[i]);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(bars.a_full(ring.slot));
        PROF_MARK(3);
        ring.advance(kAStages);
      }
      walk.advance();
    }
  }
  if (pidx == 0) PROF_FLUSH(2);
}

// =========================================================== epilogue
// Team 0 = warps 4..11.  Layers whose producer warps have nothing to do (L.epi2: every chunk raw and TMA-fed — these
// layers are short on MMAs per tile and bound by this role) add warps 12..19 as team 1: the same (lane quarter, MMA
// tile) assignment, the odd 32-column blocks, their own staging blocks, the same statistics rows.
// The last tile of layers WITH producer work (L.tail2): warps 12..19 arrive here when their patches are done
// (tail_helper) and take the team-1 share of that tile only.
template <int N, typename T, bool kPair>
__device__ __forceinline__ void epilogue_role(const ConvLayer& L, const ConvSched<N>& S, const ConvBars<N>& bars,
                                              uint32_t tmem, uint8_t* smem, int t_step, bool epi_team2,
                                              bool tail_helper PROF_PARAM) {
  using Cfg = ConvCfg<N>;
  constexpr int kRow = Cfg::kRow;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  float* bias_s = reinterpret_cast<float*>(smem + Cfg::kOffBias);
  float* tstat = reinterpret_cast<float*>(smem + Cfg::kOffTstat);
  const int team = (epi_team2 || tail_helper) ? 1 : 0;
  const int nteams0 = L.epi2 ? 2 : 1, nepi0 = nteams0 * kEpiThreads;  // teams / threads on every tile
  const bool tail2 = L.tail2 != 0;
  const int ew = team ? warp - (4 + kEpiWarps) : warp - 4;   // 0..7
  const int q = ew & 3;              // TMEM lane quarter owned by this warp (== warp % 4)
  // full tiles: one warpgroup per 128-row MMA tile; half tiles: both warpgroups drain the one MMA tile, warpgroup h
  // taking the 32-column blocks with (cb & 1) == h (a warp may only touch the TMEM lane quarter warp % 4)
  const int mt = S.two_mt ? ew >> 2 : 0;
  const int et = team ? kEpiThreads + (tid - 32 * (4 + kEpiWarps)) : tid - 128;          // 0..255 (team 0), 256..511
  const int n_off = S.n_off, n_full = L.n_full;
  if (!tail_helper) {
    const float* bias_g = L.bias + size_t(t_step) * L.bias_tstride + n_off;
    for (int i = et; i < kRow; i += nepi0) bias_s[i] = i < N ? bias_g[i] : 0.f;
    for (int i = et; i < kEpiWarps * kRow; i += nepi0) tstat[i] = 0.f;
    named_bar_sync(2, nepi0);
  }
  const int su = L.out_su;  // channel pairs per statistics entry (1, 2, 4 or 8)
  const int m = q * 32 + lane, g = m >> 3, r = m & 7;
  const bool act = L.out_mode == kOutAct;
  const bool do_stats = (L.out_stats != nullptr) && act;
  const bool has_res = (L.resid != nullptr) && act;
  const bool use_tma = N >= 32 && act;  // (N = 16 has no staging blocks)
  // staging blocks (2 KB, 512-byte aligned for the 64B swizzle).  Team 1: the third patch stage, which a producer-free
  // layer does not use (N <= 128); N = 256 has only two: the tail of the allocation + the unused GroupNorm table
  uint32_t stage_s = smem_u32(smem + Cfg::kOffStage) + uint32_t(ew) * 2048;
  if (team) {
    if constexpr (N >= 256) {
      stage_s = ew < 7 ? smem_u32(smem + Cfg::kOffStage) + uint32_t(kEpiWarps + ew) * 2048
                       : ((smem_u32(smem + Cfg::kOffTable) + 511u) & ~511u);
    } else {
      stage_s = ((smem_u32(smem + Cfg::kOffA) + 2u * kAStageBytes + 511u) & ~511u) + uint32_t(ew) * 2048;
    }
  }
  const int H = L.H, W = L.W, TH = S.TH;
  const uint32_t lane_base = tmem + (uint32_t(q * 32) << 16);
  const uint32_t run_addr = lane_base + Cfg::kStatCol0 + mt * N;  // running sums (kStatsInTmem)
  if (Cfg::kStatsInTmem && do_stats && !tail_helper) {
    uint32_t z[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) z[j] = 0u;
    for (int cb = team; cb < Cfg::kNcb; cb += nteams0) tmem_st32(run_addr + cb * 32, z);  // (N = 64: full tiles only)
    tmem_st_wait();
  }
  // a helper starts at the CTA's last tile: its accumulator stage / parity and its position follow from the tile count
  const int epi_begin = tail_helper ? S.tile_end - 1 : S.tile_begin;
  StageRing acc{(epi_begin - S.tile_begin) % S.nacc, ((epi_begin - S.tile_begin) / S.nacc) & 1};
  TileWalk walk(S.tile_first + (epi_begin - S.tile_begin) * kTileStep<kPair>, L, kTileStep<kPair>);
  // fp16 storage: values beyond +-65504 are stored saturated AND reported through the context's overflow flag, so that
  // the host can fail loudly / re-run in the bf16 mode instead of returning a silently clipped image
  constexpr bool kOverflowCheck = Cvt<T>::kFmt == 0;
  float vmax = 0.f;
  PROF_DECL;
  for (int tile = epi_begin; tile < S.tile_end; ++tile) {
    // teams on this tile, and the 32-column blocks of this warp: full tiles — one warpgroup per 128-row MMA tile, team t
    // takes blocks t, t + nteams, ...; half tiles — both warpgroups (h = ew >> 2) of a team drain the one MMA tile,
    // blocks h + 2 t, + 2 nteams, ...
    const bool helped = tail2 && tile + 1 == S.tile_end;
    const int nteams = (L.epi2 != 0 || helped) ? 2 : 1, nepi = nteams * kEpiThreads;
    const int cb_first = S.two_mt ? team : (ew >> 2) + 2 * team, cb_step = S.two_mt ? nteams : 2 * nteams;
    const int stat_bar = helped ? 3 : 2;  // (the helpers may already wait on theirs while team 0 still uses barrier 2)
    if (helped) {
      // Hand-over: everything team 0 did on earlier tiles — bias / statistics rows initialised, the previous tile's
      // statistics flushed, its running TMEM sums stored — happens before the helpers touch the same rows and columns
      if (tail_helper) {
        named_bar_sync(4, 2 * kEpiThreads);
        tc_fence_after();
      } else {
        tc_fence_before();
        __threadfence_block();
        named_bar_arrive(4, 2 * kEpiThreads);
      }
    }
    const int b = walk.b, ty = walk.ty, tx = walk.tx;
    const int x = tx * kTileW + r, y = ty * TH + mt * 16 + g;
    const bool valid = y < H && x < W;
    const bool all_valid = __all_sync(0xffffffffu, valid);
    // phase layers: b is a virtual image (image * 4 + py * 2 + px) and (y, x) a low-resolution position whose output
    // pixel is (2y + py, 2x + px) of the 2H x 2W tensor
    const int ph = L.phases > 1 ? (b & 3) : 0, b_img = L.phases > 1 ? (b >> 2) : b;
    const uint32_t pix = L.phases > 1 ? uint32_t((b_img * 2 * H + 2 * y + (ph >> 1)) * 2 * W + 2 * x + (ph & 1))
                                      : uint32_t((b * H + y) * W + x);  // < 2^31 pixels per tensor
    const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(L.resid) +
                                                     (size_t(pix) * n_full + n_off) * 2);
    uint8_t* const orow = reinterpret_cast<uint8_t*>(L.out) + (size_t(pix) * n_full + n_off) * 2;
    uint4 rq[4];  // identity residual of the next 32 channels, fetched before it is needed
    if (has_res) {
#pragma unroll
      for (int k = 0; k < 4; ++k) rq[k] = ldg16_pred(rp + cb_first * 4 + k, valid);
      // pull this lane's residual row of the NEXT tile into L2 while this tile is drained (the loads
      // above then mostly hit L2 instead of exposing HBM latency on the epilogue's critical path)
      const TileWalk next = walk.peek_next();
      const int nx = next.tx * kTileW + r, ny = next.ty * TH + mt * 16 + g;
      if (tile + 1 < S.tile_end && ny < H && nx < W) {
        const uint8_t* np = reinterpret_cast<const uint8_t*>(L.resid) +
                            (size_t(uint32_t((next.b * H + ny) * W + nx)) * n_full + n_off) * 2;
#pragma unroll
        for (int k = 0; k < N * 2; k += 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(np + k));
      }
    }
    mbar_wait(bars.acc_full(acc.slot), acc.phase);
    PROF_MARK(0);
    if (et == 0 && tile + 1 == S.tile_end) PROF_TS4(3);
    tc_fence_after();
    const uint32_t taddr = lane_base + acc.slot * S.acc_cols + mt * Cfg::kAccStride;
#pragma unroll 1
    for (int cb = cb_first; cb < Cfg::kNcb; cb += cb_step) {
      uint32_t raw[32];
      tmem_ld32(taddr + cb * 32, raw);
      tmem_ld_wait();
      PROF_MARK(3);
      float v[32];
      const float4* b4 = reinterpret_cast<const float4*>(bias_s + cb * 32);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 bb = b4[j];
        v[4 * j + 0] = __uint_as_float(raw[4 * j + 0]) + bb.x;
        v[4 * j + 1] = __uint_as_float(raw[4 * j + 1]) + bb.y;
        v[4 * j + 2] = __uint_as_float(raw[4 * j + 2]) + bb.z;
        v[4 * j + 3] = __uint_as_float(raw[4 * j + 3]) + bb.w;
      }
      if (act) {
        if (has_res) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint32_t w4[4] = {rq[k].x, rq[k].y, rq[k].z, rq[k].w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 f = Cvt<T>::unpack(w4[e]);
              v[k * 8 + e * 2] += f.x;
              v[k * 8 + e * 2 + 1] += f.y;
            }
          }
          if (cb + cb_step < Cfg::kNcb) {
#pragma unroll
            for (int k = 0; k < 4; ++k) rq[k] = ldg16_pred(rp + (cb + cb_step) * 4 + k, valid);
          }
        }
        if constexpr (kOverflowCheck) {  // largest magnitude about to be stored as fp16 (one FMNMX3 per two values)
          float cbmax = 0.f;
#pragma unroll
          for (int j = 0; j < 32; j += 2) cbmax = fmaxf(cbmax, fmaxf(fabsf(v[j]), fabsf(v[j + 1])));
          if (cbmax > 65504.f) {  // (rare) clamp what is stored AND what enters the statistics: everything downstream
#pragma unroll              // stays finite; the flag tells the host that the result is not the network's output
            for (int j = 0; j < 32; ++j) v[j] = fminf(fmaxf(v[j], -65504.f), 65504.f);
          }
          vmax = fmaxf(vmax, cbmax);
        }
        PROF_MARK(4);
        if (use_tma) {
          // stage the warp's 32 px x 32 ch block (64B-swizzled rows), then one bulk tensor store:
          // full 64-byte segments per pixel instead of 32 scattered 16-byte writes per instruction
          if (lane == 0) bulk_wait_read0();  // previous store has drained the staging block
          __syncwarp();
          PROF_MARK(5);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint32_t dst = stage_s + uint32_t(lane) * 64 + uint32_t((k ^ ((lane >> 1) & 3)) * 16);
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(dst),
                         "r"(Cvt<T>::pack_store(v[k * 8 + 0], v[k * 8 + 1])), "r"(Cvt<T>::pack_store(v[k * 8 + 2], v[k * 8 + 3])),
                         "r"(Cvt<T>::pack_store(v[k * 8 + 4], v[k * 8 + 5])), "r"(Cvt<T>::pack_store(v[k * 8 + 6], v[k * 8 + 7]))
                         : "memory");
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_4d(ph == 0 ? &L.out_map : &L.out_map_ph[ph - 1], stage_s, n_off + cb * 32, tx * kTileW,
                         ty * TH + mt * 16 + q * 4, b_img);
            bulk_commit_group();
          }
        } else if (valid) {
          uint4* op = reinterpret_cast<uint4*>(orow + cb * 64);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            uint4 u;
            u.x = Cvt<T>::pack_store(v[k * 8 + 0], v[k * 8 + 1]);
            u.y = Cvt<T>::pack_store(v[k * 8 + 2], v[k * 8 + 3]);
            u.z = Cvt<T>::pack_store(v[k * 8 + 4], v[k * 8 + 5]);
            u.w = Cvt<T>::pack_store(v[k * 8 + 6], v[k * 8 + 7]);
            op[k] = u;
          }
        }
        PROF_MARK(6);
        if (do_stats) {
          // in place: v[2p] <- pair sum, v[2p+1] <- pair sum of squares (zero for masked rows)
          if (all_valid) {
#pragma unroll
            for (int p = 0; p < 16; ++p) {
              const float a = v[2 * p], c2 = v[2 * p + 1];
              v[2 * p] = a + c2;
              v[2 * p + 1] = fmaf(a, a, c2 * c2);
            }
          } else {
#pragma unroll
            for (int p = 0; p < 16; ++p) {
              const float a = valid ? v[2 * p] : 0.f, c2 = valid ? v[2 * p + 1] : 0.f;
              v[2 * p] = a + c2;
              v[2 * p + 1] = fmaf(a, a, c2 * c2);
            }
          }
          if (Cfg::kStatsInTmem) {
            // per-lane running sums in spare TMEM columns; lanes are reduced when the sample changes
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              uint32_t run[16];
              tmem_ld16(run_addr + cb * 32 + hh * 16, run);
              tmem_ld_wait();
#pragma unroll
              for (int j = 0; j < 16; ++j) run[j] = __float_as_uint(__uint_as_float(run[j]) + v[hh * 16 + j]);
              tmem_st16(run_addr + cb * 32 + hh * 16, run);
            }
          } else {
            // entry layout per 32 channels: float [pair][2]; a unit of `su` pairs accumulates into
            // the entry of its first pair (the others stay zero), so consumers need not know `su`
            float* trow = tstat + ew * kRow + cb * 32;
            if (su == 1) {
              const float tot = warp_transpose_reduce<32>(v, lane);
              trow[lane] = tot;
            } else if (su == 2) {
              float w[16];
#pragma unroll
              for (int u = 0; u < 8; ++u) {
                w[2 * u] = v[4 * u] + v[4 * u + 2];
                w[2 * u + 1] = v[4 * u + 1] + v[4 * u + 3];
              }
              const float tot = warp_transpose_reduce<16>(w, lane);
              const int idx = lane >> 1;
              if ((lane & 1) == 0) trow[(idx >> 1) * 4 + (idx & 1)] = tot;
            } else if (su == 4) {
              float w[8];
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                w[2 * u] = (v[8 * u] + v[8 * u + 2]) + (v[8 * u + 4] + v[8 * u + 6]);
                w[2 * u + 1] = (v[8 * u + 1] + v[8 * u + 3]) + (v[8 * u + 5] + v[8 * u + 7]);
              }
              const float tot = warp_transpose_reduce<8>(w, lane);
              const int idx = lane >> 2;
              if ((lane & 3) == 0) trow[(idx >> 1) * 8 + (idx & 1)] = tot;
            } else {
              float w[4];
#pragma unroll
              for (int u = 0; u < 2; ++u) {
                float a0 = 0.f, a1 = 0.f;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  a0 += v[16 * u + 2 * j];
                  a1 += v[16 * u + 2 * j + 1];
                }
                w[2 * u] = a0;
                w[2 * u + 1] = a1;
              }
              const float tot = warp_transpose_reduce<4>(w, lane);
              const int idx = lane >> 3;
              if ((lane & 7) == 0) trow[(idx >> 1) * 16 + (idx & 1)] = tot;
            }
          }
        }
        PROF_MARK(7);
      } else if (L.out_mode == kOutPosterior) {
        // final conv inside the sampler: this thread holds eps of one pixel (C = out_c <= 8 channels).  p_sample in
        // registers: x0 = clamp(a x - b eps), mean, + sigma z (z injected or the pixel's Philox blocks), fp32 state
        // updated in place, and the next step's network input rewritten — diffusion.py:157-190, 173
        if (valid && cb == 0) {
          const PostStep ps = L.post[t_step];
          const int C = L.out_c;
          const size_t HWs = size_t(H) * W, o0 = (size_t(b) * C * H + y) * W + x;
          float zv[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
          if (ps.add_noise) {
            const float* nz = L.args->noise;
            if (nz != nullptr) {
              nz += size_t(ps.z_block) * L.B * C * HWs;
#pragma unroll
              for (int c = 0; c < 8; ++c)
                if (c < C) zv[c] = nz[o0 + c * HWs];
            } else {
              philox_pixel_normals(zv, C, L.args->seed, uint32_t(t_step), L.args->image0 + b, uint32_t(y * W + x));
            }
          }
          float xp[8];
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            xp[c] = 0.f;
            if (c < C) {
              xp[c] = post1(L.x_state[o0 + c * HWs], v[c], zv[c], ps.k);
              L.x_state[o0 + c * HWs] = xp[c];
            }
          }
          if constexpr (sizeof(T) == 2) {   // channels [0, P) of the packed input (pack_pixel's layout): x_t, then 0
            T* dst = reinterpret_cast<T*>(L.xin) + (size_t(b) * HWs + size_t(y) * W + x) * 16;
            const uint32_t w0 = Cvt<T>::pack(xp[0], xp[1]), w1 = Cvt<T>::pack(xp[2], xp[3]);
            if (C <= 4) *reinterpret_cast<uint2*>(dst) = make_uint2(w0, w1);
            else *reinterpret_cast<uint4*>(dst) = make_uint4(w0, w1, Cvt<T>::pack(xp[4], xp[5]), Cvt<T>::pack(xp[6], xp[7]));
          }
        }
      } else {  // fp32 NCHW, first out_c channels (final conv -> eps)
        if (valid && cb == 0) {
          float* o = reinterpret_cast<float*>(L.out);
#pragma unroll
          for (int c = 0; c < 8; ++c)
            if (c < L.out_c) o[((size_t(b) * L.out_c + c) * H + y) * W + x] = v[c];
        }
      }
    }
    if (Cfg::kStatsInTmem && do_stats) tmem_st_wait();
    tc_fence_before();
    __syncwarp();
    if (lane == 0 && !tail_helper) mbar_arrive(bars.acc_empty(acc.slot));  // (nobody waits for the last tile's)
    PROF_MARK(1);
    acc.advance(S.nacc);
    walk.advance();
    if (do_stats) {
      const bool flush = !Cfg::kStatsInTmem || (tile + 1) % L.group == 0;
      if (flush) {
        if (Cfg::kStatsInTmem) {
          for (int cb = cb_first; cb < Cfg::kNcb; cb += cb_step) {
            uint32_t run[32];
            float fv[32];
            tmem_ld32(run_addr + cb * 32, run);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              fv[j] = __uint_as_float(run[j]);
              run[j] = 0u;
            }
            tmem_st32(run_addr + cb * 32, run);
            const float tot = warp_transpose_reduce<32>(fv, lane);
            tstat[ew * kRow + cb * 32 + lane] = tot;
          }
          tmem_st_wait();
        }
        // warps in fixed order, then order-independent 64-bit fixed-point atomics: the statistics
        // (and therefore every activation) are bitwise reproducible run to run
        named_bar_sync(stat_bar, nepi);
        // every warp total is converted to fixed point BEFORE the warps are added: integer addition is associative, so
        // the CTA's contribution does not depend on how the same 32-pixel warp blocks are grouped into tiles (full / half
        // tiles, split-N) — the tile shape may follow the batch size without changing a single bit of the result
        for (int i = et; i < N; i += nepi) {
          const float sc = (i & 1) ? L.out_sq_scale : float(kStatScale);  // entry layout [pair][2]: sum, sum of squares
          long long tsum = 0;
#pragma unroll
          for (int w8 = 0; w8 < kEpiWarps; ++w8) tsum += __float2ll_rn(tstat[w8 * kRow + i] * sc);
          atomicAdd(L.out_stats + size_t(b_img) * n_full + n_off + i, static_cast<unsigned long long>(tsum));
        }
        if (tile + 1 < S.tile_end) named_bar_sync(stat_bar, nepi);  // (the rows are rewritten by the next tile)
      }
    }
    PROF_MARK(2);
  }
  if (kOverflowCheck && vmax > 65504.f && L.flags != nullptr) atomicOr(L.flags, 1u);
  // outstanding bulk tensor stores of this warp (waiting only for their shared-memory READS — the writes are flushed
  // at grid end anyway — measured no faster: profiles/r2/ab_tail.log)
  if (lane == 0) bulk_wait_all0();
  if (et == 0) PROF_TS(6);  // epilogue of the last tile done, stores complete
  if (et == 0) PROF_FLUSH(1);
  (void)et;
}

template <int N, typename T, bool kPair>
__global__ void __launch_bounds__(kConvThreads, 1)
conv_gemm_kernel(const __grid_constant__ ConvLayer L, int t_step) {
  using Cfg = ConvCfg<N>;
  PROF_T0;
  constexpr int kASlots = Cfg::kASlots;
  constexpr int kTStep = kTileStep<kPair>;
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const ConvBars<N> bars{smem_u32(smem + Cfg::kOffBar)};
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + Cfg::kOffTmem);
  const uint32_t crank = kPair ? cluster_ctarank() : 0u;  // 0 = leader (issues the MMAs), 1 = peer

  // The tensor maps are constants of the launch: fetch them now, so that the first patch load after the launch
  // dependency resolves (and the first tile's stores) do not start with a descriptor miss.
  if (warp == 1) {
    if (lane < kMaxSrc && L.src[lane].ptr != nullptr && L.a_tma != 0) {
      prefetch_tensormap(&L.in_map[lane]);
      if (L.a_tma == 1) prefetch_tensormap(&L.in_map_c[lane]);
    }
    if (lane == 8 && N >= 32 && L.out_mode == kOutAct) prefetch_tensormap(&L.out_map);
    if (lane >= 9 && lane < 12 && L.phases > 1) prefetch_tensormap(&L.out_map_ph[lane - 9]);
  }
  if (tid == 0) {
    for (int s = 0; s < kASlots; ++s) {
      mbar_init(bars.a_full(s), kProdWarps);
      mbar_init(bars.a_empty(s), 1);
      mbar_init(bars.raw_full(s), 1);
      mbar_init(bars.pa_full(s), 1);
    }
    for (int s = 0; s < Cfg::kBStages; ++s) {
      mbar_init(bars.b_full(s), 1);
      mbar_init(bars.b_empty(s), 1);
      mbar_init(bars.pb_full(s), 1);
    }
    for (int s = 0; s < Cfg::kNumAccMax; ++s) {
      mbar_init(bars.acc_full(s), 1);
      mbar_init(bars.acc_empty(s), L.epi2 ? 2 * kEpiWarps : kEpiWarps);
      mbar_init(bars.pacc_empty(s), 1);
    }
    mbar_init_fence();
  }
  if (warp == 0) tmem_alloc<Cfg::kTmemCols, kPair>(smem_u32(tmem_slot));
  tc_fence_before();
  __syncthreads();
  // both CTAs' barriers and TMEM exist before any remote arrive / pair MMA.  Only the two MMA warps ever touch the other
  // CTA (relay arrives, cta_group::2 MMAs and commits): every thread just ARRIVES here, the MMA warps wait before their
  // loop and everyone else before the closing cluster barrier — the loader and the producers of a CTA start earlier
  // (tools/timeline.py: entry -> prologue done 1.4 us as a pair, 0.6 us alone; profiles/r2/ab_defer_csync.log)
  if (kPair) cluster_arrive();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  if (kPair && warp == 0) cluster_wait();
  if (kPair && tid == 0) {
    // the pair MMA writes the same TMEM address in both CTAs: the two allocations must agree (they do: one CTA per
    // SM, one allocation per CTA); a mismatch would corrupt results silently, so fail loudly instead
    uint32_t ra, other;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(smem_u32(tmem_slot)), "r"(crank ^ 1u));
    asm volatile("ld.shared::cluster.u32 %0, [%1];" : "=r"(other) : "r"(ra) : "memory");
    if (other != tmem) asm volatile("trap;");
  }
  // Programmatic dependent launch: the next layer's CTAs may become resident (and run the prologue
  // above) as soon as SMs drain; everything that reads or writes activations / statistics waits here
  // for the previous launch to complete.  The weight loader (warp 1) only touches constant data.
  if (tid == 0) PROF_TS(0);  // prologue done (barriers, TMEM)
  asm volatile("griddepcontrol.launch_dependents;");
  // (the loader and the producer warps first fetch constants — weights, GroupNorm gamma / beta — and wait in their roles)
  const bool epi_team2 = L.epi2 != 0 && warp >= 4 + kEpiWarps;  // (layers without producer work)
  const bool is_producer = (warp == 2 || warp == 3 || warp >= 4 + kEpiWarps) && !epi_team2;
  bool epi_role = (warp >= 4 && warp < 4 + kEpiWarps) || epi_team2;
  bool tail_helper = false;  // producer warps 12..19 after their own work: second epilogue team for the CTA's last tile
  if (warp != 1 && !is_producer) asm volatile("griddepcontrol.wait;" ::: "memory");
  if (tid == 0) PROF_TS(1);  // previous launch complete

  // contiguous, balanced range of tiles for this CTA: consecutive tiles share the sample (GroupNorm
  // table stays valid) and their halos (L2 locality).
  // The unit of assignment is a group of L.group consecutive tiles of one image: running statistics
  // are reduced per group, so every partial sum is computed identically whatever the batch size or
  // the position of the image in the batch (results are bitwise independent of how a batch is sharded).
  // Pair mode: the unit of work is a PAIR of x-neighbouring tiles (2k, 2k + 1) — tiles_x is even — of which CTA r
  // computes tile 2k + r; [tile_begin, tile_end) then counts pairs and the CTA walks every second tile.
  const int tgroup = L.group;
  const int ngroups = (L.ntiles / kTStep) / tgroup;
  // Split-N (L.nsplit > 1, low-resolution layers whose tile count would leave most SMs idle): CTA
  // `part` computes output channels [part*N, part*N + N) of the n_full-wide layer for its tiles.
  const int nsplit = L.nsplit;
  const int part = int(blockIdx.x) % nsplit;  // (split-N layers are never paired)
  const int nclusters = int(gridDim.x / kTStep) / nsplit, cid = int(blockIdx.x / kTStep) / nsplit;
  const int tq = ngroups / nclusters, tr = ngroups - tq * nclusters;
  const int unit_begin = cid * tq + (cid < tr ? cid : tr);
  const int my_units = tq + (cid < tr ? 1 : 0);
  ConvSched<N> S;
  S.tile_begin = unit_begin * tgroup;
  S.tile_end = S.tile_begin + my_units * tgroup;
  S.tile_first = S.tile_begin * kTStep + int(crank);  // (pairs: CTA r computes tile 2k + r)
  S.first = TileWalk(S.tile_first, L, kTStep);
  S.crank = crank;
  // Tile shape.  Full tiles are 32 x 8 pixels = two 128-row MMA tiles sharing every weight stage.  Half tiles (16 x 8, one
  // MMA tile; low-resolution N >= 128 layers run as CTA pairs): twice the CTAs per layer, half the patch to load and
  // normalise per CTA, and the accumulator takes N instead of 2N TMEM columns, so that N = 256 is double-buffered too.
  S.TH = L.tile_h;
  S.two_mt = S.TH == kTileH;
  S.nacc = S.two_mt ? Cfg::kNumAcc : Cfg::kNumAccMax;
  S.acc_cols = S.two_mt ? Cfg::kAccCols : Cfg::kAccStride;
  S.blob = uint32_t(L.ncg) * (kPair ? N / 2 : N) * 16;
  S.gblob = uint32_t(L.ncg) * uint32_t(L.n_full) * 16;
  S.taps_per_stage = int(Cfg::kBStageBytes / S.blob) < kMaxTaps ? int(Cfg::kBStageBytes / S.blob) : kMaxTaps;
  S.n_off = part * N;
  S.nG = L.nG;
  S.nR = L.nR;

  if (warp == 0) {
    mma_role<N, T, kPair>(L, S, bars, tmem, smem PROF_ARG);
  } else if (warp == 1) {
    loader_role<N, T, kPair>(L, S, bars, smem);
  } else if (!epi_role) {
    producer_role<N, T, kPair>(L, S, bars, smem PROF_ARG);
    // Tail help (L.tail2): the epilogue of a CTA's LAST tile has no MMAs left to hide behind — the tensor pipe of the SM
    // idles until the launch ends (3 - 9 us per layer, tools/timeline.py).  Producer warps 12..19 have finished by then
    // and share warps 4..11's TMEM lane quarters: they join as a second team for that one tile.
    if (L.tail2 != 0 && warp >= 4 + kEpiWarps && S.tile_end > S.tile_begin) {
      tail_helper = true;
      epi_role = true;
    }
  }
  if (epi_role) epilogue_role<N, T, kPair>(L, S, bars, tmem, smem, t_step, epi_team2, tail_helper PROF_ARG);

  tc_fence_before();
  if (kPair && warp != 0) cluster_wait();  // (the opening barrier's wait, see above)
  __syncthreads();
  if (kPair) cluster_sync_all();  // neither CTA frees its TMEM / exits while the pair's MMAs or commits may still touch it
  if (tid == 0) PROF_TS(7);
  if (warp == 0) tmem_dealloc<Cfg::kTmemCols, kPair>(tmem);
}

}  // namespace fdsr
