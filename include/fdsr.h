/* libfdsr — B200 (sm_100a) implementation of the FastDiffSR T-step conditional sampling path.
 *
 * C ABI, no C++ / torch types.  The reference is pure Python and has no native interface to
 * mirror, so every entry point below cites the reference code it replaces (paths relative to
 * FastDiffSR/ in the reference tree).
 *
 * Conventions
 *   - every function returns 0 on success or a negative FDSR_E_* code; nothing throws;
 *     fdsr_last_error() returns a human-readable message for the last failure on that context
 *   - "dev" pointers are CUDA device pointers owned by the caller, valid until the stream work
 *     enqueued by the call has completed; "host" pointers are ordinary host memory
 *   - C = out_channel is the number of image bands (1..8; 3 for RGB).  All image tensors are fp32 NCHW
 *     (B,C,H,W), the reference's layout, and uint8 images are HWC (B,h,w,C); H and W must be
 *     multiples of 2^(n_levels-1): 8 for the FastDiffSR UNet (three stride-2 levels,
 *     model/fastdiffsr_modules/unet.py:77-83), 32 for the SR3 baseline (five)
 *   - calls are asynchronous with respect to the host (enqueue on `stream` and return) unless
 *     stated; a context is single-owner, not thread-safe, bound to the device that was current
 *     at fdsr_create
 */
#ifndef FDSR_H_
#define FDSR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FDSR_OK 0
#define FDSR_E_INVALID -1   /* bad argument / unsupported configuration */
#define FDSR_E_CUDA -2      /* a CUDA runtime call failed */
#define FDSR_E_STATE -3     /* call order violated (weights / schedule not loaded) */
#define FDSR_E_NOTFOUND -4  /* unknown tensor / layer name */
#define FDSR_E_OVERFLOW -5  /* fp16 mode: an activation left the fp16 range (stored saturated); use FDSR_DTYPE_BF16 */

#define FDSR_DTYPE_FP16 0   /* fp16 operands + activations, fp32 accumulate (tcgen05 kind::f16).  Activation stores
                               saturate at +-65504 and raise an overflow flag (fdsr_check_overflow) */
#define FDSR_DTYPE_BF16 1   /* bf16 activations (fp32 exponent range: safe for a trained network's un-normalised residual
                               stream), fp32 accumulate.  Operands: swish(GroupNorm(x)) -- bounded -- is rounded to fp16
                               and multiplied with fp16 weights; raw inputs (1x1 residual / up / down convs) bf16 x bf16 */
#define FDSR_DTYPE_FP32 2   /* parity mode: fp32 activations, weights and accumulation on the CUDA cores (same fused
                               layer plan; eps relative L2 <= 1e-4 against the reference; ~60x slower) */

#define FDSR_MAX_LEVELS 8

#define FDSR_MODEL_FASTDIFFSR 0 /* which_model_G = "fastdiffsr": model/fastdiffsr_modules (noise-level FiLM, CLAM/SLAM) */
#define FDSR_MODEL_SR3 1        /* which_model_G = "ddpm": the SR3 comparison baseline, model/ddpm_modules (time
                                   embedding, SelfAttention); it predicts the image itself (no res2img) */

typedef struct fdsr_ctx fdsr_ctx;

/* UNet hyper-parameters: opt['model']['unet'] consumed by define_G (model/networks.py:82-119)
 * and UNet.__init__ (model/fastdiffsr_modules/unet.py:224-297). */
typedef struct fdsr_config {
  int32_t in_channel;     /* 2 * out_channel: cat[cond, x_t] */
  int32_t out_channel;    /* C, the image bands: 1..8 (3 = RGB) */
  int32_t inner_channel;  /* 64 */
  int32_t norm_groups;    /* 32 */
  int32_t n_levels;       /* len(channel_multiplier) */
  int32_t channel_mults[FDSR_MAX_LEVELS];  /* level widths inner_channel * channel_mults[l] must each be 64, 128 or
                                              256 (e.g. 64 * [1, 2, 4, 4]); any other width, 192 included, is
                                              FDSR_E_INVALID */
  int32_t res_blocks;     /* 2 */
  int32_t dtype;          /* FDSR_DTYPE_* */
  int32_t model;          /* FDSR_MODEL_* (networks.py:84-91) */
  int32_t attn_levels;    /* FDSR_MODEL_SR3: bit l set = the ResnetBlocks of resolution level l carry SelfAttention,
                             i.e. (image_size >> l) is in attn_res (ddpm_modules/unet.py:184, 211); mid[0] always does */
} fdsr_config;

/* Replaces UNet.__init__ + GaussianDiffusion.__init__ (diffusion.py:80-99): builds the layer plan.  Channel rule:
 * in_channel == 2 * out_channel and 1 <= out_channel <= 8 (both models); anything else is FDSR_E_INVALID.
 * The network input is packed as one 16-channel NHWC tensor: with P = 4 for C <= 4 and P = 8 otherwise, x_t occupies
 * channels [0, C), cond [P, P + C), every other channel is 0 (C = 3: [x0 x1 x2 0 | c0 c1 c2 0 | 0 x 8]); the stem
 * weights are permuted to match the reference's cat([cond, x_t]) order. */
int fdsr_create(const fdsr_config* cfg, fdsr_ctx** out);
int fdsr_destroy(fdsr_ctx* ctx);
const char* fdsr_last_error(const fdsr_ctx* ctx);
/* Library-level message for failures that have no context (fdsr_create). */
const char* fdsr_global_error(void);

/* Replaces netG.load_state_dict (model/model.py:148-160).  `names[i]` is the reference state_dict
 * key ("denoise_fn.downs.1.res_block.block1.block.3.weight", ...), `host_ptrs[i]` a contiguous
 * fp32 HOST array in the reference layout (conv OIHW, linear [out,in]), `numels[i]` its element
 * count (checked).  Keys of never-executed tensors (the dead 1x1 `.conv`, unet.py:212, and the 12
 * schedule buffers) are accepted and ignored.  Synchronous.  Repacks into the kernels' operand
 * layout; must be called before fdsr_set_schedule. */
int fdsr_load_weights(fdsr_ctx* ctx, const char* const* names, const float* const* host_ptrs,
                      const int64_t* numels, int32_t n);

/* The same from DEVICE memory (SURVEY 8(b): netG.to('cuda') weights need not bounce through the caller's host
 * memory): `dev_ptrs[i]` is a contiguous fp32 device array of numels[i] elements, borrowed for the duration of the
 * call; copies are ordered after prior work on `stream`.  Synchronous. */
int fdsr_load_weights_dev(fdsr_ctx* ctx, const char* const* names, const float* const* dev_ptrs,
                          const int64_t* numels, int32_t n, void* stream);

/* Replaces GaussianDiffusion.set_new_noise_schedule (diffusion.py:109-155): derives every table
 * from the T betas in float64 exactly as the reference does, and precomputes the per-step FiLM
 * bias vectors (noise level depends on t only, diffusion.py:169-170; unet.py:22-54, 242-248).
 * Synchronous.  Re-entrant (the reference calls it for 'train' and again for 'val'). */
int fdsr_set_schedule(fdsr_ctx* ctx, const double* betas, int32_t T);
/* Copies one derived table (name as registered by the reference: "betas", "alphas_cumprod",
 * ..., "posterior_mean_coef2", or "sqrt_alphas_cumprod_prev" which has T+1 entries) to host. */
int fdsr_get_table(fdsr_ctx* ctx, const char* name, double* out_host, int32_t capacity);

/* Sizes / (re)allocates the activation workspace for this shape.  Implicit in the calls below.  The allocation only
 * ever grows, so the captured graphs of previously used shapes stay valid.
 * Deviation from SURVEY 8(b), which sketched `size_t fdsr_workspace_bytes(ctx, B, H, W)` with a caller-provided
 * workspace: the context owns its workspace (captured CUDA graphs hold pointers into it), so sizing is split into
 * fdsr_reserve (allocate for a shape) + fdsr_workspace_bytes (bytes the current shape uses). */
int fdsr_reserve(fdsr_ctx* ctx, int32_t B, int32_t H, int32_t W);
size_t fdsr_workspace_bytes(const fdsr_ctx* ctx);

/* Replaces UNet.forward as called from p_mean_variance (diffusion.py:169-173): eps for step t,
 * noise_level = sqrt_alphas_cumprod_prev[t+1].  cond, x_t: (B,C,H,W) dev; eps_out: (B,C,H,W) dev. */
int fdsr_unet_forward(fdsr_ctx* ctx, const float* cond_dev, const float* xt_dev, int32_t t,
                      float* eps_out_dev, int32_t B, int32_t H, int32_t W, void* stream);

/* Replaces p_sample (diffusion.py:157-190) given eps: x0 = clamp(a_t x - b_t eps), mean, + sigma_t z.
 * z_dev may be NULL for t == 0.  In-place allowed (x_prev_dev == xt_dev).  numel: a positive multiple of C. */
int fdsr_posterior_step(fdsr_ctx* ctx, const float* xt_dev, const float* eps_dev, const float* z_dev,
                        int32_t t, float* x_prev_dev, int64_t numel, void* stream);

/* Replaces GaussianDiffusion.super_resolution / p_sample_loop (diffusion.py:192-231), batch-safe.
 *   cond_dev  (B,C,H,W) bicubic conditioning in [-1,1]
 *   noise_dev (T,B,C,H,W) injected Gaussian noise in the reference's draw order (x_T, then z for
 *             t=T-1..1), or NULL to draw from the built-in counter-based generator with `seed`
 *   sr_out_dev (B,C,H,W) = clamp(x_0,-1,1)/2 + cond   (res2img, diffusion.py:275-281)
 *   trace_out_dev NULL, or (B, 1+n_frames, C, H, W): per sample, res2img(cond) followed by
 *             res2img of x after every step with t % (1 | T/10) == 0 — the continous=True output. */
int fdsr_sample(fdsr_ctx* ctx, const float* cond_dev, const float* noise_dev, uint64_t seed,
                float* sr_out_dev, float* trace_out_dev, int32_t B, int32_t H, int32_t W,
                void* stream);
int32_t fdsr_trace_frames(const fdsr_ctx* ctx); /* 1 + n_frames for the current schedule */

/* Tiled sampling of B canvases of (C,H,W), any H, W >= 8 with H*W < 2^32 (FastDiffSR model only): overlapping tiles
 * of one shared chain.  Every step, each tile's eps (the network on the tile's window [cond | x_t]; every tile is its
 * own image for GroupNorm) is blended into one canvas-wide eps, and one posterior update moves the canvas-wide x_t.
 *   Grid, per axis of length L with tile size t (tile_h / tile_w: multiples of 8, >= 8) and overlap o (>= 0):
 *     t_e = min(t, 8*floor(L/8));  o_e = min(o, t_e - 8);  s = t_e - o_e;
 *     starts = i*s for every i >= 0 with i*s < L - t_e, then L - t_e (the last tile is flush with the far edge).
 *   Global tile order: canvas, then row start, then column start (all ascending).
 *   Weights: tile pixel (i, j) weighs r_y(i) * r_x(j), r(i) = min(i+1, t_e-i, o_e+1) (an integer, exact in fp32 for
 *     o_e < 4096).  Per canvas pixel, over the covering tiles in global order, in fp32 with round-to-nearest:
 *     n_k = w_k / sum(w);  eps = n_1 eps_1 + n_2 eps_2 + ... (the sum starts from the first term, so a pixel covered
 *     by one tile gets that tile's eps exactly);  x_{t-1} = the posterior update of fdsr_posterior_step.
 *   Noise is drawn per canvas pixel: built-in = the generator of fdsr_sample at (seed, image offset + b, y*W + x,
 *     step); injected = noise_dev (T,B,C,H,W) in fdsr_sample's draw order.  Canvas b is image fdsr_set_image_offset + b.
 *   cond_dev, sr_out_dev and trace_out_dev are as in fdsr_sample, with the canvas shape.
 *   Evaluation: the n_tiles = B * tiles_y * tiles_x tiles go through the UNet in n_chunks = ceil(n_tiles / tile_batch)
 *     calls of Bc = ceil(n_tiles / n_chunks) tiles each (the last chunk is padded with repeats of its last tile), so the
 *     activation workspace is fdsr_reserve(Bc, t_e_y, t_e_x), independent of the canvas; the canvas x_t and the
 *     per-tile eps store (n_chunks * Bc * C * t_e_y * t_e_x floats) live in a separate grow-only context allocation.
 *   A canvas that is exactly one tile gives fdsr_sample's bits; with o = 0 on a canvas the tiles partition, the result
 *   equals fdsr_sample of the crops (with the noise cropped alike); tile_batch does not change the result.
 *   Plain stream launches (no graph capture); the graphs cached by fdsr_sample are neither used nor evicted (a chunk
 *   shape that grows the workspace drops them, like any larger fdsr_sample shape).  fp16 mode: check
 *   fdsr_check_overflow as after fdsr_sample.  FDSR_E_INVALID: SR3 model, H or W < 8, H*W >= 2^32, bad tile sizes,
 *   overlap < 0, tile_batch < 1, B outside 1..65535, null cond / sr_out. */
int fdsr_sample_tiled(fdsr_ctx* ctx, const float* cond_dev, const float* noise_dev, uint64_t seed,
                      float* sr_out_dev, float* trace_out_dev, int32_t B, int32_t H, int32_t W,
                      int32_t tile_h, int32_t tile_w, int32_t overlap, int32_t tile_batch, void* stream);

/* One tiled sampling job split over the `world` ranks of a group (one process and context per GPU): every rank samples
 * its share of the tiles of the same B canvases, and the gathered result equals fdsr_sample_tiled of the same inputs
 * bit for bit, for any world size.
 *   The rule.  All ranks pass identical arguments (cond, noise or seed, image offset, canvas and tile sizes, overlap);
 *     tile_batch may differ per rank.
 *   - Tile ownership: the n = B * tiles_y * tiles_x tiles in their global order (canvas, row start, column start) are
 *     split into contiguous ranges; rank r owns [floor(r n / world), floor((r+1) n / world)).  The range is empty iff
 *     the two bounds are equal, which happens only when world > n.
 *   - Update region U_r: the union of the windows of rank r's tiles.  Every step rank r computes the eps of its own tiles,
 *     receives the eps of every other rank's tile whose window intersects U_r, and blends and updates exactly the
 *     pixels of U_r (fdsr_sample_tiled's arithmetic).  Pixels a neighbour also updates get identical bits on both ranks
 *     (same x_t, the same eps in the same order, the same noise), so x_t is never exchanged: only eps, once per step.
 *   - Exchange plan (fdsr_tiled_plan): for each ordered pair q -> r, q sends one contiguous range of its own tile slots,
 *     from the first to the last of its tiles r needs (a superset: every slot in it holds q's valid eps), into the same
 *     slots of r's store.  With heavy overlaps (o_e >= t_e / 2) a pixel lies under 3 or more tile rows and r may need
 *     tiles of ranks that are not adjacent to it; the plan covers them.
 *   - Output: a pixel belongs to the rank that owns its first covering tile in global order (these owners partition the
 *     canvas).  Each rank writes sr_out and the trace frames at its pixels and +0.0 everywhere else, so an integer sum
 *     of the int32 bit patterns over the ranks (all_reduce SUM of the int32 view) rebuilds the exact bits, -0.0 included.
 *   - Why the bits match: by induction over the steps, x_t on U_r equals the single-GPU x_t.  A tile's eps depends only
 *     on x_t in its window (and not on the chunk it is evaluated in: tile_batch does not change the result), every own
 *     window lies in U_r, every foreign window lies in its owner's update region, and the blend reads each covering
 *     tile in global order.
 *
 * Host only, needs no context or GPU: the exchange plan of `rank`.  out_host[0 .. 5 + 4 world):
 *   n_tiles, t_e_y, t_e_x, own_lo, own_hi, then for each peer q = 0 .. world-1: send_lo, send_hi (the slots rank sends
 *   to q), recv_lo, recv_hi (the slots rank receives from q); empty ranges and q == rank are 0, 0.  recv of r from q
 *   equals send of q to r.  Returns the entry count, or FDSR_E_INVALID (message in fdsr_global_error) for the arguments
 *   fdsr_sample_tiled rejects, world < 1, rank outside 0..world-1, a null out_host or cap < 5 + 4 world. */
int64_t fdsr_tiled_plan(int32_t B, int32_t H, int32_t W, int32_t tile_h, int32_t tile_w, int32_t overlap,
                        int32_t world, int32_t rank, int64_t* out_host, int64_t cap);

/* Moves the eps slots of one step between the ranks' stores (see fdsr_sample_tiled_part).  `step` is t (T-1 .. 0).
 * Returns 0, or nonzero to abort the sampling call. */
typedef int (*fdsr_tile_exchange_fn)(void* user, int32_t step, void* stream);

/* Rank `rank`'s part of the split job above (arguments as in fdsr_sample_tiled).
 *   eps_store_dev: caller-owned n_tiles x C x t_e_y x t_e_x fp32, indexed by global tile, so that the exchange can send
 *     from it and receive into it directly.  The call writes its own slots.
 *   exchange: called once per step on the host, after the own tiles' eps have been enqueued into the store on `stream`
 *     and before the blend is enqueued.  It must order its transfers after prior work on `stream` and make `stream`
 *     wait for their completion (for example NCCL send / recv of the plan's ranges).  A nonzero return aborts the call
 *     with FDSR_E_INVALID.  NULL is accepted only when the plan of this rank has no transfers (for example world 1).
 *   A rank with an empty range runs no UNet but still calls exchange every step, so that collectives match.
 *   sr_out_dev / trace_out_dev: the rank's pixels, +0.0 elsewhere.  Launches per call: 2 + T (chunks (1 + UNet ops) + 1)
 *     + trace frames + 1, with chunks = ceil(own tiles / tile_batch).
 *   FDSR_E_INVALID: everything fdsr_sample_tiled rejects, a null eps_store_dev, world < 1, rank outside 0..world-1, a
 *   NULL exchange when the plan has transfers. */
int fdsr_sample_tiled_part(fdsr_ctx* ctx, const float* cond_dev, const float* noise_dev, uint64_t seed,
                           float* sr_out_dev, float* trace_out_dev, int32_t B, int32_t H, int32_t W, int32_t tile_h,
                           int32_t tile_w, int32_t overlap, int32_t tile_batch, int32_t rank, int32_t world,
                           float* eps_store_dev, fdsr_tile_exchange_fn exchange, void* user, void* stream);

/* Tiled sampling of scenes with nodata: fdsr_sample_tiled (same arguments and checks) with a validity mask
 * valid_dev, a (B,H,W) uint8 array at the canvas resolution, nonzero = valid; all bands of a pixel share it.
 *   Active tile: a tile of fdsr_sample_tiled's grid (same t_e, o_e, starts and global order) whose window holds at
 *     least one valid pixel.  Only active tiles go through the UNet.
 *   Chunking over the n_active active tiles in global order: n_chunks = ceil(n_active / tile_batch) UNet calls of
 *     Bc = ceil(n_active / n_chunks) tiles (the last one padded with repeats); the eps store holds active tiles only.
 *   Blend and update: per pixel over its *active* covering tiles in global order, with fdsr_sample_tiled's weights,
 *     normalisation and fp32 round-to-nearest, the sums starting from the first active term.  A pixel with no active
 *     covering tile is not updated; such a pixel is always invalid (every tile covering a valid pixel is active).
 *   Noise: unchanged, drawn per canvas pixel from the same generator or noise_dev.
 *   Output: valid pixels get fdsr_sample_tiled's res2img(x); invalid pixels get cond_dev, bit for bit.  Trace frames
 *     follow the same rule.
 *   Hence: when every tile is active (an all-valid mask among others) the valid pixels are fdsr_sample_tiled's bits;
 *   with overlap 0 on a canvas the tiles partition and a mask invalid exactly on whole tiles, the valid pixels equal
 *   fdsr_sample of the remaining crops (noise cropped alike); tile_batch does not change the result.
 *   The tile flags are computed on the device (one block per tile) and read back once: the call synchronises `stream`
 *   once, before it enqueues the sampling.  Launches: 1 + fdsr_sample_tiled's count with n_tiles replaced by n_active,
 *   i.e. 3 + T * (n_chunks * (1 + UNet launches) + 1) + trace frames.  A canvas with no active tile runs no UNet and
 *   returns cond (trace frames too).  FDSR_E_INVALID: everything fdsr_sample_tiled rejects, a null valid_dev, more than
 *   2^31 - 1 tiles. */
int fdsr_sample_tiled_masked(fdsr_ctx* ctx, const float* cond_dev, const uint8_t* valid_dev, const float* noise_dev,
                             uint64_t seed, float* sr_out_dev, float* trace_out_dev, int32_t B, int32_t H, int32_t W,
                             int32_t tile_h, int32_t tile_w, int32_t overlap, int32_t tile_batch, void* stream);

/* fp16 mode only (always FDSR_OK otherwise): synchronises `stream`, then returns FDSR_E_OVERFLOW if any activation
 * stored since the last check had left the fp16 range (it was stored saturated, so nothing downstream is inf / NaN,
 * but the image is not the network's output), and clears the flag.  fdsr_super_resolve_u8 performs this check itself;
 * callers of the asynchronous fdsr_sample call it when they synchronise. */
int fdsr_check_overflow(fdsr_ctx* ctx, void* stream);

/* Position of subsequent batches in the job: `first_image` is the global index of image 0 of the next fdsr_sample /
 * fdsr_super_resolve_u8 batches.  The built-in generator's counter is (position in the image, GLOBAL image index,
 * step), so image k of a job receives the same noise whether it is sampled alone, inside a batch, or by another rank:
 * a batch sharded over N ranks (rank r passes the index of its first image) equals the single-rank result bit for bit.
 * Sticky; default 0.  Read from device memory by the captured graph (no re-capture).
 * The generator: Philox4x32-10 keyed by the 64-bit seed, counter (pixel index y*W + x, low 32 bits of the global image
 * index, step stream, (0x5eed + high 32 bits of the image index) ^ f), four normals per evaluation by Box-Muller.  Band c
 * of a pixel takes normal c mod 4 of block c div 4, where block 0 has f = 0 and block 1 has f = 0x80000000; so bands
 * 0-2 receive the same values for every C. */
int fdsr_set_image_offset(fdsr_ctx* ctx, uint64_t first_image);

/* Host-buffer convenience for callers without device memory management (the end-to-end path that
 * bench.py times): uint8 LR (B,h,w,C) host -> PIL-exact bicubic -> sampling -> fp32 SR (B,C,H,W)
 * host.  Copies go through context-owned pinned staging buffers.  Synchronous. */
int fdsr_super_resolve_u8(fdsr_ctx* ctx, const uint8_t* lr_host, int32_t B, int32_t h, int32_t w,
                          int32_t H, int32_t W, const float* noise_dev, uint64_t seed,
                          float* sr_out_host, void* stream);

/* The same, pipelined for throughput: two slots.  submit enqueues H2D, bicubic, sampling and — on an internal copy stream —
 * the D2H of one batch into `slot` (0 or 1) and returns; wait blocks until that slot's result is in its pinned buffer,
 * copies it to sr_out_host and reports FDSR_E_OVERFLOW if the fp16 guard fired for that batch.  With one batch submitted
 * ahead, the copies and the host-side memcpy of batch i overlap the sampling of batch i+1. */
int fdsr_super_resolve_u8_submit(fdsr_ctx* ctx, int32_t slot, const uint8_t* lr_host, int32_t B, int32_t h, int32_t w,
                                 int32_t H, int32_t W, const float* noise_dev, uint64_t seed, void* stream);
int fdsr_super_resolve_u8_wait(fdsr_ctx* ctx, int32_t slot, float* sr_out_host);

/* New at the boundary (the reference precomputes it offline with PIL, data/prepare_data_mfe_dm.py
 * :30-40): bit-exact Pillow BICUBIC resize of uint8 HWC images (horizontal pass, uint8 rounding,
 * vertical pass; 22-bit fixed-point taps; each band resized as Pillow resizes an 'L' image), then optional /255*2-1
 * to fp32 NCHW (data/util.py:66-75).
 *   lr_dev (B,h,w,C) u8;  out_u8_dev (B,H,W,C) u8 or NULL;  cond_out_dev (B,C,H,W) fp32 or NULL */
int fdsr_bicubic_u8(fdsr_ctx* ctx, const uint8_t* lr_dev, int32_t B, int32_t h, int32_t w,
                    int32_t H, int32_t W, uint8_t* out_u8_dev, float* cond_out_dev, void* stream);

/* PSNR accumulators for the sharded evaluation loop (sr_mfe.py:315-356, core/metrics.py:16-42,
 * 94-101): per image, quantise both tensors like tensor2img (clamp [-1,1] -> uint8) and add the
 * squared error sum to sse_out_dev[b] (double, B entries) of (B,C,H,W) tensors.  PSNR = 10 log10(255^2 * CHW / sse). */
int fdsr_sse_u8(fdsr_ctx* ctx, const float* a_dev, const float* b_dev, int32_t B, int32_t H,
                int32_t W, double* sse_out_dev, void* stream);

/* Device-side evaluation metrics replacing the host block of sr_mfe.py:315-356 (skimage compare_mse /
 * compare_psnr / compare_ssim(multichannel=True) and core/metrics.py:88-93 calculate_ergas on
 * Metrics.tensor2img uint8 images, core/metrics.py:16-42).  a = the evaluated image (SR or bicubic),
 * b = HR, both (B,C,H,W) fp32 in [-1,1] on the device.  out_dev: B x 4 doubles (mse, psnr, ssim, ergas).
 * MSE / PSNR over the C*H*W values; SSIM: 7x7 uniform window, sample covariance, K1 = .01, K2 = .03, data_range 255,
 * 3-pixel crop, mean over the C channels; ERGAS: 100 sqrt(mse / mean(a)^2 / C) / ergas_scale. */
int fdsr_metrics_u8(fdsr_ctx* ctx, const float* a_dev, const float* b_dev, int32_t B, int32_t H, int32_t W,
                    double ergas_scale, double* out_dev, void* stream);

/* 16-bit imagery.  The white level max_value = M (1..65535) is the sample value that maps to +1: 65535 for 16-bit
 * data, 4095 for 12-bit, 2047 for 11-bit, 10000 for reflectance scaled by 10^4.
 *
 * uint16 (B,h,w,C) dev -> Pillow-exact BICUBIC resize of each band as Pillow resizes an 'I;16' image (Pillow 12.2):
 * the bounds and normalised double weights of fdsr_bicubic_u8 before its fixed-point step; horizontal pass, then
 * vertical, with a uint16 intermediate; per sample ss = 0.0, ss = ss + double(p) * k in float64, every multiply and add
 * rounded on its own; v = ss >= 0 ? floor(ss + 0.5) : -floor(-ss + 0.5); stored byte by byte as Pillow stores I;16,
 * lo = CLIP8(v % 256), hi = CLIP8(v >> 8).  So v < 0 gives 0, 0..65535 gives v, and v > 65535 gives
 * 65280 + v % 256, not 65535 (Pillow's store quirk, reproduced so that an sr_ folder written by Pillow and the
 * conditioning rebuilt here are the same bits).  A uint16 image is always resized this way, even when its values fit
 * in 8 bits: with M = 255 the result is not fdsr_bicubic_u8's, which uses 22-bit fixed point.
 *   out_u16_dev (B,H,W,C) the resized levels (not clamped to max_value), or NULL;
 *   cond_out_dev (B,C,H,W) fp32 = (min(v, max_value) / max_value) * 2 - 1 (fp32, each step rounded to nearest), or NULL.
 * FDSR_E_INVALID: max_value outside 1..65535, a null lr_dev, both outputs null, B, h, w, H or W < 1. */
int fdsr_bicubic_u16(fdsr_ctx* ctx, const uint16_t* lr_dev, int32_t B, int32_t h, int32_t w, int32_t H, int32_t W,
                     int32_t max_value, uint16_t* out_u16_dev, float* cond_out_dev, void* stream);
/* fdsr_metrics_u8 at white level max_value: both images are quantised to levels 0..M by
 * rint(((clamp(x, -1, 1) + 1) / 2) * M) in fp32 (ties to even); PSNR = 10 log10(M^2 / mse); SSIM with data_range M
 * (C1 = (0.01 M)^2, C2 = (0.03 M)^2); ERGAS as in fdsr_metrics_u8.  max_value = 255 gives fdsr_metrics_u8's bits.
 * FDSR_E_INVALID: max_value outside 1..65535, null pointers, B, H or W < 1. */
int fdsr_metrics_u16(fdsr_ctx* ctx, const float* a_dev, const float* b_dev, int32_t B, int32_t H, int32_t W,
                     int32_t max_value, double ergas_scale, double* out_dev, void* stream);
/* fdsr_metrics_u16 over the valid pixels only: valid_dev (B,H,W) uint8, nonzero = valid (all bands share it).
 *   MSE and the ERGAS mean run over the C |V| values of the valid pixels V; PSNR = 10 log10(M^2 / MSE);
 *   SSIM = the mean, over the C channels and the cropped-interior positions whose whole 7x7 window is valid, of
 *   fdsr_metrics_u16's SSIM map.  No such window: SSIM is NaN.  |V| = 0: all four are NaN.
 *   An all-valid mask gives fdsr_metrics_u16's bits (fdsr_metrics_u8's at max_value = 255).  The SSIM accumulator
 *   limit of fdsr_metrics_u16 (about 8.4 M band-pixels, DESIGN 4.6) applies unchanged.
 * FDSR_E_INVALID: as fdsr_metrics_u16, and a null valid_dev. */
int fdsr_metrics_masked(fdsr_ctx* ctx, const float* a_dev, const float* b_dev, const uint8_t* valid_dev, int32_t B,
                        int32_t H, int32_t W, int32_t max_value, double ergas_scale, double* out_dev, void* stream);

/* ---- test / profiling hooks (not part of the drop-in surface) ---- */
/* Number of activation tensors of the current plan and their names ("downs.0", "downs.1.h", ...). */
int32_t fdsr_debug_num_tensors(const fdsr_ctx* ctx);
const char* fdsr_debug_tensor_name(const fdsr_ctx* ctx, int32_t i);
/* Converts activation tensor `name` of the last fdsr_unet_forward (NHWC 16-bit) to fp32 NCHW. */
int fdsr_debug_read_tensor(fdsr_ctx* ctx, const char* name, float* out_dev, int64_t capacity,
                           int32_t* C, int32_t* H, int32_t* W, void* stream);
/* Per-op profiling of one UNet evaluation on the context's current buffers (call after a forward
 * or sample at the shape of interest): runs the ops `reps` times with a CUDA-event pair around
 * each op's launch(es) on `stream`, writes the mean milliseconds per op to ms_out_host (for reps >= 4 the
 * mean of the last reps/2 repetitions: the first half warms the GPU up to its sustained clocks) and returns
 * the number of ops.  Synchronous.  Op names / algorithmic conv FLOPs (at the reserved shape) for
 * turning the times into TFLOP/s: */
int32_t fdsr_debug_num_ops(const fdsr_ctx* ctx);
const char* fdsr_debug_op_name(const fdsr_ctx* ctx, int32_t i);
double fdsr_debug_op_flops(const fdsr_ctx* ctx, int32_t i);
/* The multiply-adds the op really executes: equal to the algorithmic figure except for the three nearest-upsample convs,
 * which run as four 2x2 phase convs on the low-resolution input (4/9 of the nine-tap MACs). */
double fdsr_debug_op_flops_executed(const fdsr_ctx* ctx, int32_t i);
/* The schedule conv op `i` is launched with at the current shape (16-bit modes, after a forward at that shape; host
 * only), as the launch computes it: out_host[0..16] = N (per CTA), pair (CTA pairs), tile_h (32, or 16 = half tiles),
 * nsplit (split-N parts), group (tiles per statistics group), grid (CTAs), ntiles, the largest tile count of one CTA,
 * epi2, tail2, nR, nG (patch ring stages), phases (4 = phase-decomposed upsample), a_tma, whether some CTA's range
 * holds tiles of two images, whether some CTA's range holds tiles of two phases of one image, and the K chunk count.
 * Returns the number of fields written (17); cap must be at least that. */
int fdsr_debug_op_schedule(fdsr_ctx* ctx, int32_t i, int32_t* out_host, int32_t cap);
int fdsr_debug_profile_unet(fdsr_ctx* ctx, int32_t t, int32_t reps, float* ms_out_host, int32_t cap,
                            void* stream);
/* Role-level cycle counters of one conv op (only populated by -DFDSR_PROFILE builds of the library,
 * used by tools/role_profile.py): out_host[(cta*5 + role)*8 + slot], role 0 = MMA issuer, 1 = epilogue,
 * 2 = producer, 3 = timeline (cycles since kernel entry of: prologue done, previous launch complete, GroupNorm table
 * built, first patch landed, first MMA, last MMA issued, epilogue done, exit), 4 = anchor {SM id, the SM's clock at
 * kernel entry, %globaltimer at entry}.  Re-runs op `op` on the current buffers; returns the number of entries.
 * Synchronous. */
int fdsr_debug_role_cycles(fdsr_ctx* ctx, int32_t op, int32_t t, int64_t* out_host, int32_t cap, void* stream);
/* The same counters of EVERY conv op inside a running UNet evaluation (tools/timeline.py): `reps` evaluations back to
 * back, launched as the sampler launches them (programmatic dependent launch); out_host[op][sm][role][slot] of the
 * last one (cap >= num_ops * num_sms * 40 entries).  Consecutive launches on one SM share its clock, so
 * first-MMA(op k+1) - last-MMA(op k) is the tensor pipe's idle time between two layers.  Returns the number of ops. */
int fdsr_debug_timeline(fdsr_ctx* ctx, int32_t t, int32_t reps, int64_t* out_host, int64_t cap, void* stream);
/* Fills out_dev (B,C,H,W) with the N(0,1) values the built-in generator hands the sampler for step stream
 * `stream_id` (T for x_T, t for the z of step t) of images first_image .. first_image+B-1 under `seed`: lets tests
 * check the distribution (moments, Kolmogorov-Smirnov) and reproduce a built-in-noise sample through the
 * injected-noise path bit for bit. */
int fdsr_debug_noise(fdsr_ctx* ctx, float* out_dev, int32_t B, int32_t H, int32_t W, uint64_t seed,
                     uint64_t first_image, int32_t stream_id, void* stream);
/* Number of CUDA-graph captures of the sampling loop so far (cache misses of the per-shape graph cache). */
int64_t fdsr_graph_captures(const fdsr_ctx* ctx);
/* Kernel launches enqueued by this context so far (library kernels only). */
int64_t fdsr_launch_count(const fdsr_ctx* ctx);
/* Algorithmic conv FLOPs (2*MAC, padding counted) of one UNet forward at the reserved shape. */
double fdsr_unet_flops(const fdsr_ctx* ctx);
/* 1 = capture the T-step loop into a CUDA graph per shape (default), 0 = plain stream launches. */
int fdsr_set_use_graph(fdsr_ctx* ctx, int32_t enable);

#ifdef __cplusplus
}
#endif
#endif /* FDSR_H_ */
