// Host/device shared description of one fused convolution launch.
//
// Every heavy layer of the UNet (3x3 conv, stride-2 conv, nearest-up conv, 1x1 residual conv,
// all with optional GroupNorm+Swish on their input, FiLM/bias on their output, residual add and
// GroupNorm statistics of their output) is ONE launch of conv_gemm_kernel described by a
// ConvLayer: a list of K-chunks (<= 64 input channels each, from one source tensor), each with a
// list of taps (a shifted view of the resident input patch x a packed weight blob).
#pragma once
#include <cstdint>
#include <cuda.h>  // CUtensorMap (type only; the encoder is fetched through cudaGetDriverEntryPoint)

namespace fdsr {

constexpr int kMaxChunks = 24;
constexpr int kMaxTaps = 9;
constexpr int kMaxSrc = 3;

// Output tile: 32 rows x 8 columns of output pixels = two 128-row MMA tiles (16x8 each).
constexpr int kTileH = 32;
constexpr int kTileW = 8;
constexpr int kPatchW = kTileW + 2;           // input patch pitch in positions
constexpr int kPatchH = kTileH + 2;
constexpr int kPatchPos = kPatchW * kPatchH;  // 340 positions
constexpr int kPlanePos = 341;                // odd => conflict-free 16B stores across channel groups
constexpr int kPlaneBytes = kPlanePos * 16;
constexpr int kPlaneBytesTma = 344 * 16;      // plane pitch when the planes are written by TMA (a_tma = 2): bulk tensor
                                              // copies need a 128-byte aligned shared-memory destination
// TMA-fed layers keep the patch pixel-major instead: 128 bytes (64 channels) per position,
// 128B-swizzled exactly as a SWIZZLE_128B tensor load of the NHWC source leaves it.
constexpr int kPatchBytesSw = kPatchPos * 128;  // 43,520
// one A stage holds either layout.  341 x 128 B: stage s starts (5 s mod 8) rows into the 1024-byte
// swizzle period, which the in-place transform accounts for (the MMA unit and TMA both swizzle on
// absolute shared-memory address bits, so they agree on any 128-byte-aligned base).
constexpr int kAStageBytes = 8 * kPlaneBytes;  // 43,648
static_assert(kPatchBytesSw <= kAStageBytes && kAStageBytes % 128 == 0, "A stage too small");

enum ConvMode : int32_t {
  kModeNormal = 0,  // stride-1 3x3 (or 1x1 via a single centre tap), zero padding 1
  kModeUp2x = 1,    // nearest x2 upsample folded into the gather, then stride-1 3x3
  kModeS2D = 2,     // stride-2 3x3 expressed as 2x2 taps over space-to-depth parity planes
};

enum OutMode : int32_t {
  kOutAct = 0,        // 16-bit NHWC activation (+ optional identity residual, + pair statistics)
  kOutEpsNCHW = 1,    // fp32 NCHW, first `out_c` channels only (final conv -> eps: the fdsr_unet_forward hook)
  kOutPosterior = 2,  // final conv inside the sampler: eps stays in registers, the epilogue does the whole p_sample
                      // update (diffusion.py:157-190) on the fp32 x_t state in place and writes the next step's
                      // 16-bit network input channels (diffusion.py:173) — no eps tensor, no separate kernels
};

// Per-call arguments of the sampler that live in DEVICE memory, so that one captured CUDA graph per
// (B, H, W, injected-noise?, trace?) serves every seed, image offset, noise tensor and trace tensor.
struct SampleArgs {
  uint64_t seed;         // Philox key
  uint64_t image0;       // global index of the first image of this batch
  const float* noise;    // (T,B,C,H,W) injected noise, or null: built-in generator
  float* trace;          // (B, frames, C, H, W), or null
};
// posterior coefficients of one step (diffusion.py:140-155 tables as fp32, like the reference's registered buffers)
struct PostCoef {
  float a, b, c1, c2, sigma;
};
struct PostStep {
  PostCoef k;
  int32_t z_block;    // block of the injected noise tensor holding this step's z (1 + steps already done)
  int32_t add_noise;  // 0 for t == 0
  int32_t pad_[1];
};

struct ConvChunk {
  int32_t src;        // index into ConvLayer::src
  int32_t c0;         // first channel inside the source tensor
  int32_t gn;         // 1: GroupNorm+Swish with scale/shift table entries [vc0, vc0+64); 2: GroupNorm only (no activation)
  int32_t vc0;        // channel offset on the virtual (concatenated) GroupNorm axis
  int32_t ntaps;
  int32_t ring;       // patch ring of this chunk: 0 = full stages, 1 = 32 KB centre-box stages (ConvLayer::nR > 0)
  int32_t center;     // 1: TMA-fed raw chunk whose only tap is the centre one: staged as a dense 32x8 box (no halo)
  int32_t w_off;      // byte offset of this chunk's first tap blob inside the layer's weights
  int32_t parity;     // kModeS2D: pa*2 + pb of the space-to-depth plane this chunk reads (TMA-fed form), else 0
  int32_t tap_pos[kMaxTaps];  // A-operand position offset of each tap (dy*kPatchW + dx)
};

struct ConvSrc {
  const void* ptr;      // NHWC 16-bit
  const unsigned long long* stats;  // [B][C/2][2] fixed-point (sum, sum of squares) per channel pair, or null
  int32_t C;
  int32_t H, W;         // spatial size of the source tensor
};

struct ConvLayer {
  // TMA descriptor of the 16-bit NHWC output tensor, dims {C, W, H, B}, box {32 ch, 8, 4, 1},
  // 64B swizzle: each epilogue warp stores its 32 px x 32 ch block with one bulk tensor copy (kOutAct, N >= 32)
  alignas(64) CUtensorMap out_map;
  // TMA descriptors of the 16-bit NHWC source tensors, dims {C, W, H, B}, box {64 ch, 10, 34, 1},
  // 128B swizzle: one bulk tensor load stages a whole (32+2)x(8+2) x 64-channel input patch,
  // out-of-image positions zero-filled (a_tma = 1; a_tma = 2: in_map[0] is the stem's 8-channel plane map)
  CUtensorMap in_map[kMaxSrc];
  CUtensorMap in_map_c[kMaxSrc];  // same tensors, box {64 ch, 8, 32, 1}: centre-only chunks (1x1 residual conv);
                                  // kModeS2D: box {64 ch, 20, 68, 1} traversed with element strides {1, 2, 2, 1}: one
                                  // load = the 10 x 34 patch of one space-to-depth parity plane of the stride-2 conv
  // phases = 4 (nearest-x2 upsample + 3x3 conv evaluated as four 2x2 convs on the low-resolution input, one per
  // output parity (py, px)): strided views of the output tensor for phases 1..3 (phase 0 uses out_map): dims
  // {C, W, H, B} of the low-resolution grid, element strides {1, 2C, 2*Wout*C, Hout*Wout*C}, base + (py*Wout + px)*C
  CUtensorMap out_map_ph[3];
  ConvSrc src[kMaxSrc];
  ConvChunk chunk[kMaxChunks];
  int32_t nchunks;
  int32_t ncg;          // 16-byte channel groups per chunk (8, or 2 for the 16-channel stem input)
  int32_t mode;         // ConvMode
  int32_t nG, nR;       // patch stages in ring 0 (full) / ring 1 (centre boxes); nR = 0: single ring
  int32_t a_tma;        // 1: input patches arrive by TMA (kModeNormal and kModeS2D, 64-channel chunks); 2: the 16-channel
                        // stem input arrives as two 8-channel TMA plane loads (no-swizzle patch layout); 0 (kModeUp2x in
                        // the nine-tap form): gathered by the producer warps
  int32_t B, H, W;      // output size
  int32_t N;            // MMA N of one CTA (16 / 64 / 128 / 256)
  int32_t n_full;       // channel width of the output tensor and of the packed weight blobs (= N * nsplit)
  int32_t nsplit;       // CTAs sharing one output tile along N (1 = none): part p owns channels [p*N, p*N+N)
  // GroupNorm over the virtual concat of src[0..nsrc) (only chunks with gn=1 use it)
  int32_t gn_C;         // virtual channels (0 = no GroupNorm in this layer)
  int32_t gn_nsrc;
  int32_t gn_groups;
  const float* gamma;   // [gn_C]
  const float* beta;    // [gn_C]
  float gn_eps;
  // epilogue
  const float* bias;    // [T or 1][N] fp32: conv bias (+ residual-conv bias) (+ FiLM vector of step t)
  int32_t bias_tstride; // floats between steps (0 when the bias does not depend on t)
  const void* resid;    // identity residual, NHWC 16-bit with N channels, or null
  void* out;            // NHWC 16-bit [B][H][W][N]  |  fp32 NCHW [B][out_c][H][W]
  unsigned long long* out_stats;  // [B][N/2][2] fixed point, or null
  float out_sq_scale;   // fixed-point scale of the sums of squares of the OUTPUT tensor (power of two, see stat_sq_scale)
  double gn_inv_sum, gn_inv_sq;  // GroupNorm input: 1 / (scale * elements per group) for the sums / sums of squares
  int32_t out_su;       // channel pairs per statistics entry (1, 2, 4, 8): coarsest unit every consumer can use
  int32_t out_mode;     // OutMode
  int32_t out_c;
  const uint8_t* weights;  // packed blobs
  int32_t pair;            // 1: launched as CTA pairs (conv_gemm_kernel<.., kPair = true>): `weights` is the half-width
  int32_t w_half;          //    layout, CTA r of a pair reads from weights + r * w_half
  int32_t phases;          // 1, or 4: tiles run over virtual images (image * 4 + phase), H/W are the low-resolution
                           // grid, every tap position is shifted by (py*kPatchW + px), weights are per phase
  int32_t epi2;            // 1: layers without producer work (every chunk raw, patches by TMA: up / down-sampling convs,
                           //    stem) turn producer warps 12..19 into a second epilogue team (odd 32-column blocks)
  int32_t tail2;           // 1: producer warps 12..19 join the epilogue of the CTA's LAST tile as a second team (layers with
                           //    producer work; the last tile's epilogue is exposed — nothing is left to overlap it with)
  int32_t tile_h;          // output rows per CTA tile: 32 (two 128-row MMA tiles) or 16 (one: "half tiles", see upload_layers)
  int32_t tiles_x, tiles_y, ntiles;
  int32_t group;           // tiles per assignment group (divides tiles_x * tiles_y)
  // kOutPosterior
  const PostStep* post;    // [T]
  float* x_state;          // fp32 NCHW (B,out_c,H,W): x_t in, x_{t-1} out (in place)
  void* xin;               // 16-bit NHWC16 network input: channels [0, out_c) receive x_{t-1} (pack_pixel's layout)
  const SampleArgs* args;
  unsigned int* flags;     // context status word: bit 0 = an fp16 activation store saturated (overflow)
  long long* prof;         // role cycle counters [grid][5 roles][8 slots] (FDSR_PROFILE builds only)
};

}  // namespace fdsr
