// libfdsr: C-ABI, context, layer plan, weight packing and launch orchestration (see include/fdsr.h).
// The plan mirrors UNet.__init__/forward of the reference (model/fastdiffsr_modules/unet.py:224-323);
// each ResnetBlock becomes two conv_gemm_kernel launches, each Down/Upsample one.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <utility>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/fdsr.h"
#include "aux_kernels.cuh"
#include "conv_kernel.cuh"
#include "conv_f32.cuh"
#include "attn_kernel.cuh"
#include "tile_kernels.cuh"

using namespace fdsr;

namespace {

thread_local std::string g_global_error;

struct HTensor {
  std::string name;
  int C = 0, level = 0;
  bool stats = false;
  int unit = 0;  // gcd (channels) of the GroupNorm units every consumer needs; 0 = no GroupNorm consumer
  size_t off = 0, stats_off = 0;  // byte offsets inside the workspace
};

struct HTap {
  int ky, kx, pos;
};
struct HChunk {
  int slot, c0, gn, vc0, parity;  // parity: -1 or pa*2+pb (space-to-depth plane)
  std::vector<HTap> taps;
  std::string wname;
  int wc0;      // first input channel inside the weight tensor
  int creal;    // real (non-padded) channels in this chunk
  int kk = 3;   // kernel size of the weight tensor (3, or 1 for res_conv / attention projections)
  // stem only: the packed network input holds x_t in channels [0, C) and cond in [P, P + C) (pack_pixel) while the
  // reference concatenates cat([cond, x]) (diffusion.py:173): perm[j] = reference input channel of packed channel j, or -1
  std::vector<int> perm;
  int wchan(int ci) const { return perm.empty() ? (ci < creal ? wc0 + ci : -1) : (ci < int(perm.size()) ? perm[ci] : -1); }
  int wchan_end() const { return perm.empty() ? wc0 + creal : *std::max_element(perm.begin(), perm.end()) + 1; }
  int nreal() const {
    if (perm.empty()) return creal;
    int n = 0;
    for (int v : perm) n += v >= 0;
    return n;
  }
};
struct HConv {
  std::string name;
  int mode = kModeNormal, N = 0, cout = 0, ncg = 8;
  int nsrc = 0, src[kMaxSrc] = {-1, -1, -1};
  int gn_C = 0, gn_nsrc = 0;
  std::string gn_name;
  std::vector<HChunk> chunks;
  std::vector<std::string> bias_names;
  std::string film_name;
  int resid = -1, out = -1, out_mode = kOutAct, out_c = 0;
  int phases = 1;            // 4: nearest-x2 upsample + 3x3 conv as four 2x2 convs on the low-resolution input (see add_up)
  int w_n0 = 0, w_rows = 0;  // this launch uses rows [w_n0, w_n0 + cout) of a weight tensor with w_rows rows (0 = cout)
  bool film_swish = false;   // FiLM vector = Linear(swish(emb)) (SR3 ResnetBlock.mlp) instead of Linear(emb)
  // device-side resources
  size_t w_off = 0;      // into weight arena
  size_t w_off2 = 0, w_bytes = 0;  // pair-capable layers: a second copy as two half-width layouts (CTA pairs), layer bytes
  bool pair_ok() const { return ncg == 8 && N >= 64 && out_mode == kOutAct; }
  size_t gamma_off = 0;  // into param arena (floats)
  size_t bias_off = 0;   // into bias arena (floats), [T][N]
};
struct HAttn {
  std::string name;
  int kind = 0;  // 0: CLAM + SLAM gates (FastDiffSR mid[0]); 1: SelfAttention core softmax(q k^T / sqrt(C)) v (SR3)
  int in = -1, out = -1, C = 0;
  int tq = -1, tk = -1, tv = -1;              // kind 1: q / k / v tensors (`out` is the un-projected attention output)
  size_t w1_off = 0, w2_off = 0, w7_off = 0;  // param arena (floats)
};
struct HOp {
  int kind;  // 0 conv, 1 attention (HAttn)
  int idx;
};

// Device memory owned by a context, freed with it.  grow(bytes) keeps the allocation when it is already large enough:
// cached graphs and tensor maps hold pointers into it.
template <typename T>
struct DevBuf {
  T* ptr = nullptr;
  size_t cap = 0;  // bytes
  DevBuf() = default;
  DevBuf(DevBuf&& o) noexcept : ptr(o.ptr), cap(o.cap) {
    o.ptr = nullptr;
    o.cap = 0;
  }
  DevBuf(const DevBuf&) = delete;
  ~DevBuf() { cudaFree(ptr); }
  operator T*() const { return ptr; }
  cudaError_t grow(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    cudaFree(ptr);
    ptr = nullptr;
    cap = 0;
    const cudaError_t e = cudaMalloc(&ptr, bytes);
    if (e == cudaSuccess) cap = bytes;
    return e;
  }
};

}  // namespace

struct fdsr_ctx {
  fdsr_config cfg{};
  int device = 0, num_sms = 0;
  std::string err;
  std::vector<HTensor> tensors;
  std::vector<HConv> convs;
  std::vector<HAttn> attns;
  std::vector<HOp> ops;
  int t_xin = -1, t_last = -1;
  // weights
  std::map<std::string, std::vector<float>> host_w;
  bool weights_loaded = false;
  DevBuf<uint8_t> d_weights;
  DevBuf<float> d_params;  // gamma/beta, clam/slam weights
  DevBuf<float> d_bias;    // per conv [T][N]
  // schedule
  int T = 0;
  std::map<std::string, std::vector<double>> tables;
  std::vector<PostCoef> post;
  // workspace
  int B = 0, H = 0, W = 0;
  DevBuf<uint8_t> d_ws;  // grow-only: the captured graphs of other shapes hold pointers into it
  size_t ws_bytes = 0;
  size_t stats_off = 0, stats_bytes = 0;
  size_t off_cond = 0, off_x = 0, off_eps = 0, off_sr = 0, off_psum = 0, off_pmax = 0, off_gate = 0,
         off_sp = 0, off_seed = 0;
  std::vector<ConvLayer> h_layers;  // passed by value as __grid_constant__ kernel parameters
  std::vector<F32Layer> f_layers;   // fp32 parity mode: the same plan for conv_f32_kernel
  std::vector<F32GnArgs> f_gn;
  std::vector<AttnParams> a_params;  // per HAttn of kind 1 (16-bit modes)
  // Test hooks, read by fdsr_create: each forces a form that the automatic choice also picks for some layer or
  // configuration, so that the tests can compare the two forms (INTEGRATION.md §2)
  bool pair = true;        // FDSR_PAIR=0: never launch CTA pairs (cta_group::2); every layer runs the single-CTA kernel
  bool half_tiles = true;  // FDSR_HALF_TILES=0: 32 x 8 tiles everywhere (the <= 64^2 wide layers then use split-N / single accumulators)
  bool split_n = true;     // FDSR_SPLIT_N=0: never split a layer's output channels over two CTAs
  bool epi2 = true;        // FDSR_EPI2=0: producer-free layers keep one epilogue team (warps 4..11)
  bool tail_help = true;   // FDSR_TAIL_HELP=0: the last tile of a CTA is drained by warps 4..11 alone
  bool resid_mma = true;   // FDSR_RESID_MMA=0: identity residuals are always added by the epilogue
  bool up_phases = true;   // FDSR_UP_PHASES=0: nearest-upsample convs gather a 2x patch and run all nine taps
  bool fused_tail = true;  // FDSR_FUSED_TAIL=0: the sampler runs pack_input / final conv -> eps / posterior as separate kernels
  bool attn_ref = false;   // FDSR_ATTN_REF=1: CUDA-core attention core in the 16-bit modes too
  DevBuf<float> d_weights32;        // fp32 parity mode weights: per conv, per chunk [tap][ci][N]
  std::vector<size_t> w32_off;      // per conv (floats)
  size_t off_gntab = 0;             // [B][kMaxGnC] float2 scratch of the fp32 mode
  int esize() const { return cfg.dtype == FDSR_DTYPE_FP32 ? 4 : 2; }
  int bands() const { return cfg.out_channel; }  // C: channels of every image tensor (cond, x_t, eps, noise, SR, u8)
  DevBuf<long long> d_prof;  // role cycle counters (FDSR_PROFILE builds)
  bool layers_dirty = true;
  // bicubic tables (cached per size pair)
  struct BicTab {
    int in, out, ksize;
    DevBuf<int> d_min, d_cnt, d_taps;
  };
  std::vector<BicTab> bic;
  DevBuf<uint8_t> d_bic_tmp;
  DevBuf<unsigned long long> d_metric;  // [B][4] integer accumulators of fdsr_metrics_u8
  // pinned staging for the host-buffer path
  // host-buffer path: two slots so that the copies of one batch overlap the sampling of the next
  struct HostSlot {
    uint8_t* h_pin = nullptr;      // pinned: [LR u8 | SR fp32 | status word]
    size_t h_pin_bytes = 0;
    DevBuf<uint8_t> d_stage;       // device: [LR u8 | cond fp32 | SR fp32 | status word]
    size_t in_b = 0, out_b = 0;
    cudaEvent_t computed = nullptr, copied = nullptr;
    bool busy = false;
  };
  static constexpr int kHostSlots = 2;
  HostSlot slot[kHostSlots];
  cudaStream_t copy_stream = nullptr;
  // graph cache
  bool use_graph = true;
  DevBuf<PostStep> d_post;         // [T] per-step posterior arguments of the fused final-conv epilogue
  ConvLayer final_fused{};         // the final conv's descriptor in kOutPosterior mode (h_layers holds the eps form)
  // Captured sampling loops, keyed on what the captured launches depend on: the shape and whether noise is injected /
  // a trace is written.  Seed, image offset and the noise / trace POINTERS are read from device memory (SampleArgs),
  // so a fresh noise tensor, a new seed or a ragged last batch followed by a full one never forces a re-capture.
  struct GraphEntry {
    int B, H, W;
    bool noise, trace;
    cudaGraphExec_t exec;
    uint64_t used;
    int64_t launches;   // kernels per replay
  };
  std::vector<GraphEntry> graphs;   // small LRU (kMaxGraphs)
  uint64_t graph_clock = 0;
  int64_t graph_captures = 0;
  uint64_t image0 = 0;              // fdsr_set_image_offset
  void drop_graphs() {
    for (auto& g : graphs) cudaGraphExecDestroy(g.exec);
    graphs.clear();
  }
  int64_t launches = 0;
  double flops_per_px = 0.0;  // conv FLOPs per full-resolution output pixel per image
  // fdsr_sample_tiled: [SampleArgs | canvas x_t (B,C,H,W) fp32 | per-tile eps store [slot][C][te_y][te_x] fp32],
  // grow-only, apart from the workspace (which only ever holds one chunk of tiles)
  DevBuf<uint8_t> d_tiled;
};

namespace {

int fail(fdsr_ctx* c, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (c) c->err = buf;
  else g_global_error = buf;
  return code;
}

// Test hooks (fdsr_ctx): "0" / "1" in the environment turn one off / on; unset or any other value keeps the default
bool env_hook(const char* name, bool dflt) {
  const char* e = getenv(name);
  return e && (e[0] == '0' || e[0] == '1') ? e[0] == '1' : dflt;
}

#define CUDA_TRY(c, expr)                                                                    \
  do {                                                                                       \
    cudaError_t e_ = (expr);                                                                 \
    if (e_ != cudaSuccess)                                                                   \
      return fail(c, FDSR_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, \
                  __LINE__);                                                                 \
  } while (0)

// The tail of every kernel launch: check it where it happens, and count it (fdsr_launch_count)
int launched(fdsr_ctx* c, cudaError_t e, const void* kernel) {
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) {
    const char* name = nullptr;
    if (cudaFuncGetName(&name, kernel) != cudaSuccess || !name) name = "kernel";
    return fail(c, FDSR_E_CUDA, "launch of %s failed: %s", name, cudaGetErrorString(e));
  }
  ++c->launches;
  return FDSR_OK;
}

template <typename... P, typename... A>
int launch(fdsr_ctx* c, void (*kernel)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, A&&... args) {
  kernel<<<grid, block, smem, st>>>(std::forward<A>(args)...);
  return launched(c, cudaSuccess, reinterpret_cast<const void*>(kernel));
}

// Replaces the buffer with a device copy of `host`, allocated `pad` bytes longer
template <typename T, typename H>
int upload(fdsr_ctx* c, DevBuf<T>& b, const std::vector<H>& host, size_t pad = 0) {
  cudaFree(b.ptr);
  b.ptr = nullptr;
  b.cap = 0;
  CUDA_TRY(c, b.grow(host.size() * sizeof(H) + pad));
  CUDA_TRY(c, cudaMemcpy(b.ptr, host.data(), host.size() * sizeof(H), cudaMemcpyHostToDevice));
  return FDSR_OK;
}

// f(Elem<T>{}) with the context's element type T: __half, __nv_bfloat16, or float (the fp32 parity mode).
// with_dtype16 serves the paths that exist for the 16-bit types only; their callers have ruled out fp32.
template <typename T>
struct Elem {
  using type = T;
};
template <typename F>
auto with_dtype16(const fdsr_ctx* c, F&& f) {
  return c->cfg.dtype == FDSR_DTYPE_BF16 ? f(Elem<__nv_bfloat16>{}) : f(Elem<__half>{});
}
template <typename F>
auto with_dtype(const fdsr_ctx* c, F&& f) {
  return c->cfg.dtype == FDSR_DTYPE_FP32 ? f(Elem<float>{}) : with_dtype16(c, f);
}

int pad_n(int cout) { return cout <= 16 ? 16 : (cout <= 64 ? 64 : (cout <= 128 ? 128 : 256)); }

constexpr int kOpScheduleFields = 17;  // fdsr_debug_op_schedule

void add_conv(fdsr_ctx* c, const HConv& k) {
  c->convs.push_back(k);
  c->ops.push_back({0, int(c->convs.size()) - 1});
}

int add_tensor(fdsr_ctx* c, const std::string& name, int C, int level, bool stats) {
  HTensor t;
  t.name = name;
  t.C = C;
  t.level = level;
  t.stats = stats;
  c->tensors.push_back(t);
  return int(c->tensors.size()) - 1;
}

std::vector<HTap> taps3x3() {
  std::vector<HTap> v;
  for (int ky = 0; ky < 3; ++ky)
    for (int kx = 0; kx < 3; ++kx) v.push_back({ky, kx, ky * kPatchW + kx});
  return v;
}

// ResnetBlock (unet.py:104-120) -> two fused conv launches. Returns the output tensor id.
int add_res(fdsr_ctx* c, const std::string& name, const std::vector<int>& srcs, int cout, int level,
            const std::string& out_name) {
  const std::string p = "denoise_fn." + name + ".res_block";
  int cin = 0;
  for (int s : srcs) cin += c->tensors[s].C;
  const int th = add_tensor(c, name + ".h", cout, level, true);
  const int to = add_tensor(c, out_name, cout, level, true);
  {
    HConv k;
    k.name = name + ".block1";
    k.N = pad_n(cout);
    k.cout = cout;
    k.nsrc = int(srcs.size());
    for (size_t i = 0; i < srcs.size(); ++i) k.src[i] = srcs[i];
    k.gn_C = cin;
    k.gn_nsrc = int(srcs.size());
    k.gn_name = p + ".block1.block.0";
    int vc = 0;
    for (size_t si = 0; si < srcs.size(); ++si)
      for (int c0 = 0; c0 < c->tensors[srcs[si]].C; c0 += 64, vc += 64)
        k.chunks.push_back({int(si), c0, 1, vc, -1, taps3x3(), p + ".block1.block.3.weight", vc, 64});
    k.bias_names = {p + ".block1.block.3.bias"};
    // FeatureWiseAffine (fastdiffsr unet.py:38-54): Linear(emb); SR3 ResnetBlock.mlp (ddpm unet.py:82-85): Linear(swish(emb))
    k.film_swish = c->cfg.model == FDSR_MODEL_SR3;
    k.film_name = k.film_swish ? p + ".mlp.1" : p + ".noise_func.noise_func.0";
    k.out = th;
    add_conv(c, k);
  }
  {
    HConv k;
    k.name = name + ".block2";
    k.N = pad_n(cout);
    k.cout = cout;
    k.src[0] = th;
    k.nsrc = 1;
    k.gn_C = cout;
    k.gn_nsrc = 1;
    k.gn_name = p + ".block2.block.0";
    for (int c0 = 0; c0 < cout; c0 += 64)
      k.chunks.push_back({0, c0, 1, c0, -1, taps3x3(), p + ".block2.block.3.weight", c0, 64});
    k.bias_names = {p + ".block2.block.3.bias"};
    if (cin != cout) {
      int vc = 0;
      for (size_t si = 0; si < srcs.size(); ++si) {
        k.src[k.nsrc] = srcs[si];
        for (int c0 = 0; c0 < c->tensors[srcs[si]].C; c0 += 64, vc += 64)
          k.chunks.push_back({k.nsrc, c0, 0, 0, -1, {{0, 0, kPatchW + 1}}, p + ".res_conv.weight", vc, 64, 1});
        ++k.nsrc;
      }
      k.bias_names.push_back(p + ".res_conv.bias");
    } else if (c->resid_mma && c->cfg.dtype != FDSR_DTYPE_FP32 && pad_n(cout) == 64) {
      // identity residual of an N = 64 layer as one more K chunk with the identity matrix as weights: x * 1 is exact
      // in fp16/bf16 and accumulates in fp32 like the epilogue's add, but the tile arrives by TMA (centre box) and
      // the epilogue — the bottleneck of these layers — neither loads nor adds it (8 extra MMAs per 72)
      k.src[k.nsrc] = srcs[0];
      for (int c0 = 0; c0 < cout; c0 += 64)
        k.chunks.push_back({k.nsrc, c0, 0, 0, -1, {{0, 0, kPatchW + 1}}, "@identity", c0, 64, 1});
      ++k.nsrc;
    } else {
      k.resid = srcs[0];
    }
    k.out = to;
    add_conv(c, k);
  }
  return to;
}

// SelfAttention of the SR3 baseline (ddpm_modules/unet.py:100-131) on tensor `in` (C channels):
//   q, k, v = three 1x1 convs with GroupNorm (no activation) fused into their prologue, weights = row blocks of
//             attn.qkv.weight (n_head = 1: chunk(3) along the channel axis);
//   o       = softmax(q k^T / sqrt(C)) v  (attn_kernel.cuh);
//   out     = 1x1 conv(o) + bias + in, with the GroupNorm statistics of the result.
int add_self_attn(fdsr_ctx* c, const std::string& name, int in, int level, const std::string& out_name) {
  const std::string p = "denoise_fn." + name + ".attn";
  const int C = c->tensors[in].C;
  int tq[3];
  const char* sfx[3] = {".attn.q", ".attn.k", ".attn.v"};
  for (int i = 0; i < 3; ++i) {
    tq[i] = add_tensor(c, name + sfx[i], C, level, false);
    HConv k;
    k.name = name + sfx[i];
    k.N = pad_n(C);
    k.cout = C;
    k.nsrc = 1;
    k.src[0] = in;
    k.gn_C = C;
    k.gn_nsrc = 1;
    k.gn_name = p + ".norm";
    for (int c0 = 0; c0 < C; c0 += 64)
      k.chunks.push_back({0, c0, 2, c0, -1, {{0, 0, kPatchW + 1}}, p + ".qkv.weight", c0, 64, 1});
    k.w_n0 = i * C;
    k.w_rows = 3 * C;
    k.out = tq[i];
    add_conv(c, k);
  }
  HAttn a;
  a.name = name;
  a.kind = 1;
  a.in = in;
  a.C = C;
  a.tq = tq[0];
  a.tk = tq[1];
  a.tv = tq[2];
  a.out = add_tensor(c, name + ".attn.o", C, level, false);
  c->attns.push_back(a);
  c->ops.push_back({1, int(c->attns.size()) - 1});
  const int to = add_tensor(c, out_name, C, level, true);
  {
    HConv k;
    k.name = name + ".attn.out";
    k.N = pad_n(C);
    k.cout = C;
    k.nsrc = 1;
    k.src[0] = a.out;
    for (int c0 = 0; c0 < C; c0 += 64)
      k.chunks.push_back({0, c0, 0, 0, -1, {{0, 0, kPatchW + 1}}, p + ".out.weight", c0, 64, 1});
    k.bias_names = {p + ".out.bias"};
    k.resid = in;
    k.out = to;
    add_conv(c, k);
  }
  return to;
}

// ResnetBlocWithAttn (ddpm_modules/unet.py:134-147): ResnetBlock, then SelfAttention when `attn`
int add_res_attn(fdsr_ctx* c, const std::string& name, const std::vector<int>& srcs, int cout, int level, bool attn) {
  if (!attn) return add_res(c, name, srcs, cout, level, name);
  const int tr = add_res(c, name, srcs, cout, level, name + ".res");
  return add_self_attn(c, name, tr, level, name);
}

// MACs per output pixel of a conv (real channels only; identity-residual chunks are bookkeeping, not convolution work).
// Algorithmic: a phase layer counts as the nine-tap conv it replaces; executed: as the four-tap convs it runs.
double conv_macs(const HConv& k, bool executed) {
  double macs = 0.0;
  for (const HChunk& ch : k.chunks)
    macs += ch.wname == "@identity" ? 0.0 : double((k.phases == 4 && !executed) ? 9 : ch.taps.size()) * ch.nreal();
  return macs;
}

int build_plan(fdsr_ctx* c) {
  const fdsr_config& g = c->cfg;
  const int inner = g.inner_channel;
  if (g.out_channel < 1 || g.out_channel > 8 || g.in_channel != 2 * g.out_channel)
    return fail(c, FDSR_E_INVALID,
                "in_channel must be 2 * out_channel with 1 <= out_channel <= 8 (conditional SR of C-band images; got "
                "in_channel=%d, out_channel=%d)", g.in_channel, g.out_channel);
  if (inner % 64 != 0) return fail(c, FDSR_E_INVALID, "inner_channel must be a multiple of 64");
  if (g.norm_groups != 32) return fail(c, FDSR_E_INVALID, "norm_groups must be 32");
  if (g.n_levels < 1 || g.n_levels > FDSR_MAX_LEVELS) return fail(c, FDSR_E_INVALID, "bad n_levels");
  if (g.model != FDSR_MODEL_FASTDIFFSR && g.model != FDSR_MODEL_SR3) return fail(c, FDSR_E_INVALID, "unknown model %d", g.model);
  const bool sr3 = g.model == FDSR_MODEL_SR3;
  // a level's tensors are allocated with its width and its convs are planned at pad_n(width) channels: the two agree
  // only for 64, 128 and 256 (a 192-wide level would be written at a 256-channel pitch)
  for (int i = 0; i < g.n_levels; ++i) {
    const int w = inner * g.channel_mults[i];
    if (g.channel_mults[i] < 1 || (w != 64 && w != 128 && w != 256))
      return fail(c, FDSR_E_INVALID,
                  "level %d: channel width inner_channel * channel_mults[%d] = %d unsupported (every level width must be "
                  "64, 128 or 256)", i, i, w);
  }
  c->t_xin = add_tensor(c, "xin", 16, 0, false);
  int level = 0, pre = inner, idx = 1;
  int cur = add_tensor(c, "downs.0", inner, 0, true);
  {
    HConv k;
    k.name = "downs.0";
    k.N = pad_n(inner);
    k.cout = inner;
    k.ncg = 2;
    k.nsrc = 1;
    k.src[0] = c->t_xin;
    // packed [x (C) | 0 | cond (C) | 0] with cond at P = 4 (C <= 4) or 8 -> reference cat([cond, x]) channels
    const int C = g.out_channel, P = C <= 4 ? 4 : 8;
    HChunk stem{0, 0, 0, 0, -1, taps3x3(), "denoise_fn.downs.0.weight", 0, P + C};
    stem.perm.assign(16, -1);
    for (int j = 0; j < C; ++j) {
      stem.perm[j] = C + j;
      stem.perm[P + j] = j;
    }
    k.chunks.push_back(stem);
    k.bias_names = {"denoise_fn.downs.0.bias"};
    k.out = cur;
    add_conv(c, k);
  }
  std::vector<int> feats{cur};
  for (int li = 0; li < g.n_levels; ++li) {
    const int cm = inner * g.channel_mults[li];
    for (int r = 0; r < g.res_blocks; ++r, ++idx) {
      const std::string nm = "downs." + std::to_string(idx);
      cur = add_res_attn(c, nm, {cur}, cm, level, sr3 && ((g.attn_levels >> li) & 1));
      feats.push_back(cur);
      pre = cm;
    }
    if (li != g.n_levels - 1) {
      const std::string nm = "downs." + std::to_string(idx++);
      const int to = add_tensor(c, nm, pre, level + 1, true);
      HConv k;
      k.name = nm;
      k.mode = kModeS2D;
      k.N = pad_n(pre);
      k.cout = pre;
      k.nsrc = 1;
      k.src[0] = cur;
      for (int pa = 0; pa < 2; ++pa)
        for (int pb = 0; pb < 2; ++pb)
          for (int c0 = 0; c0 < pre; c0 += 64) {
            HChunk ch{0, c0, 0, 0, pa * 2 + pb, {}, "denoise_fn." + nm + ".conv.weight", c0, 64};
            for (int bdy = (pa ? -1 : 0); bdy <= 0; ++bdy)
              for (int bdx = (pb ? -1 : 0); bdx <= 0; ++bdx)
                ch.taps.push_back({2 * bdy + pa + 1, 2 * bdx + pb + 1, (bdy + 1) * kPatchW + (bdx + 1)});
            k.chunks.push_back(ch);
          }
      k.bias_names = {"denoise_fn." + nm + ".conv.bias"};
      k.out = to;
      add_conv(c, k);
      cur = to;
      ++level;
      feats.push_back(cur);
    }
  }
  // mid: ResnetBlock + CLAM/SLAM, ResnetBlock (unet.py:274-279); SR3: ResnetBlock + SelfAttention, ResnetBlock
  if (sr3) {
    cur = add_res_attn(c, "mid.0", {cur}, pre, level, true);
    cur = add_res_attn(c, "mid.1", {cur}, pre, level, false);
  } else {
    const int tr = add_res(c, "mid.0", {cur}, pre, level, "mid.0.res");
    HAttn a;
    a.name = "mid.0";
    a.in = tr;
    a.C = pre;
    a.out = add_tensor(c, "mid.0", pre, level, true);
    c->attns.push_back(a);
    c->ops.push_back({1, 0});
    cur = add_res(c, "mid.1", {a.out}, pre, level, "mid.1");
  }
  idx = 0;
  for (int li = g.n_levels - 1; li >= 0; --li) {
    const int cm = inner * g.channel_mults[li];
    for (int r = 0; r < g.res_blocks + 1; ++r, ++idx) {
      const int skip = feats.back();
      feats.pop_back();
      const std::string nm = "ups." + std::to_string(idx);
      cur = add_res_attn(c, nm, {cur, skip}, cm, level, sr3 && ((g.attn_levels >> li) & 1));
      pre = cm;
    }
    if (li >= 1) {
      const std::string nm = "ups." + std::to_string(idx++);
      const int to = add_tensor(c, nm, pre, level - 1, true);
      HConv k;
      k.name = nm;
      k.N = pad_n(pre);
      k.cout = pre;
      k.nsrc = 1;
      k.src[0] = cur;
      // Upsample (unet.py:66-74): nearest x2, then conv3x3.  Output pixel (2Y+py, 2X+px) only ever sees the 2x2
      // low-resolution neighbourhood rows {Y-1+py, Y+py} x cols {X-1+px, X+px}: the three taps of a row/column that
      // fall on the same source pixel are added up front (pack_weights), so each output parity is a 2x2 conv on
      // the low-resolution tensor -- 4 instead of 9 MACs per weight, TMA-fed like every other stride-1 layer.
      // An exact identity up to the rounding of the summed weights; the fp32 parity mode keeps the nine-tap form.
      k.phases = (c->up_phases && g.dtype != FDSR_DTYPE_FP32 && pre >= 128) ? 4 : 1;
      k.mode = k.phases == 4 ? kModeNormal : kModeUp2x;
      for (int c0 = 0; c0 < pre; c0 += 64) {
        if (k.phases == 4)
          k.chunks.push_back({0, c0, 0, 0, -1,
                              {{0, 0, 0}, {0, 1, 1}, {1, 0, kPatchW}, {1, 1, kPatchW + 1}},  // (ry, rx, patch position)
                              "denoise_fn." + nm + ".conv.weight", c0, 64});
        else
          k.chunks.push_back({0, c0, 0, 0, -1, taps3x3(), "denoise_fn." + nm + ".conv.weight", c0, 64});
      }
      k.bias_names = {"denoise_fn." + nm + ".conv.bias"};
      k.out = to;
      add_conv(c, k);
      cur = to;
      --level;
    }
  }
  {
    HConv k;
    k.name = "final_conv";
    k.N = 16;
    k.cout = g.out_channel;
    k.nsrc = 1;
    k.src[0] = cur;
    k.gn_C = pre;
    k.gn_nsrc = 1;
    k.gn_name = "denoise_fn.final_conv.block.0";
    for (int c0 = 0; c0 < pre; c0 += 64)
      k.chunks.push_back({0, c0, 1, c0, -1, taps3x3(), "denoise_fn.final_conv.block.3.weight", c0, 64});
    k.bias_names = {"denoise_fn.final_conv.block.3.bias"};
    k.out_mode = kOutEpsNCHW;
    k.out_c = g.out_channel;
    add_conv(c, k);
  }
  c->t_last = cur;
  // Statistics granularity per tensor: a consumer GroupNorm with cpg channels per group over the
  // virtual concat [src0 (C0), src1] can use entries of gcd(cpg, C0) channels (cpg when un-concatenated).
  auto gcd = [](int a, int b) { while (b) { int t = a % b; a = b; b = t; } return a; };
  for (const HConv& k : c->convs) {
    if (k.gn_C == 0) continue;
    const int cpg = k.gn_C / g.norm_groups;
    const int unit = k.gn_nsrc == 2 ? gcd(cpg, c->tensors[k.src[0]].C) : cpg;
    for (int s = 0; s < k.gn_nsrc; ++s) {
      HTensor& t = c->tensors[k.src[s]];
      t.unit = t.unit ? gcd(t.unit, unit) : unit;
    }
  }
  for (HTensor& t : c->tensors)
    if (t.stats && t.unit == 0) t.stats = false;  // nobody normalises this tensor
  // sanity + algorithmic FLOPs (2*MAC, padding counted, real channels only)
  double fl = 0.0;
  for (const HConv& k : c->convs) {
    if (int(k.chunks.size()) > kMaxChunks) return fail(c, FDSR_E_INVALID, "layer %s: too many chunks", k.name.c_str());
    if (k.gn_C > kMaxGnC) return fail(c, FDSR_E_INVALID, "layer %s: GroupNorm width %d > %d", k.name.c_str(), k.gn_C, kMaxGnC);
    const int lvl = k.out >= 0 ? c->tensors[k.out].level : 0;
    fl += 2.0 * conv_macs(k, false) * k.cout / double(1 << (2 * lvl));
  }
  c->flops_per_px = fl;
  return FDSR_OK;
}

const std::vector<float>* find_w(fdsr_ctx* c, const std::string& name);

// The weight tensor [rows][cin][kk][kk] a chunk reads.  cin follows from the tensor's size, which validate_weights has
// checked against the channels the plan reads (the 256 x 256 identity has no state_dict entry).
struct WeightGeom {
  size_t rows, kk, cin;
  WeightGeom(const HConv& k, const HChunk& ch, size_t numel = 0)
      : rows(k.w_rows ? k.w_rows : k.cout), kk(ch.kk), cin(ch.wname == "@identity" ? 256 : numel / (rows * kk * kk)) {}
  size_t at(int n, int ci, int ky, int kx) const { return ((size_t(n) * cin + ci) * kk + ky) * kk + kx; }
};

// Exact element counts of every tensor the plan reads, before anything indexes into them: the C ABI is a public
// boundary that does not go through torch's strict shape check, and a state_dict of a different inner_channel /
// channel_mults must be refused by name, not read out of bounds (model/model.py:159-160 raises in the same situation).
int validate_weights(fdsr_ctx* c) {
  auto need = [&](const std::string& name, size_t numel, const char* what) -> int {
    const auto* w = find_w(c, name);
    if (!w) return fail(c, FDSR_E_NOTFOUND, "state_dict is missing %s", name.c_str());
    if (w->size() != numel)
      return fail(c, FDSR_E_INVALID, "%s: %s has %zu elements, the configured network needs %zu", what, name.c_str(),
                  w->size(), numel);
    return FDSR_OK;
  };
  const size_t inner = size_t(c->cfg.inner_channel);
  int rc;
  // conv weights: rows x (sum of the source channels this weight tensor spans) x k x k
  std::map<std::string, size_t> numel_of;
  for (const HConv& k : c->convs)
    for (const HChunk& ch : k.chunks) {
      if (ch.wname == "@identity") continue;
      const WeightGeom g(k, ch);
      size_t& n = numel_of[ch.wname];
      n = std::max(n, g.rows * ch.wchan_end() * g.kk * g.kk);
    }
  for (const auto& it : numel_of)
    if ((rc = need(it.first, it.second, "conv weight"))) return rc;
  for (const HConv& k : c->convs) {
    for (const std::string& bn : k.bias_names)
      if ((rc = need(bn, size_t(k.cout), "conv bias"))) return rc;
    if (k.gn_C) {
      if ((rc = need(k.gn_name + ".weight", size_t(k.gn_C), "GroupNorm weight"))) return rc;
      if ((rc = need(k.gn_name + ".bias", size_t(k.gn_C), "GroupNorm bias"))) return rc;
    }
    if (!k.film_name.empty()) {  // FeatureWiseAffine / ResnetBlock.mlp: Linear(inner -> cout)
      if ((rc = need(k.film_name + ".weight", size_t(k.cout) * inner, "FiLM weight"))) return rc;
      if ((rc = need(k.film_name + ".bias", size_t(k.cout), "FiLM bias"))) return rc;
    }
  }
  // noise_level_mlp / time_mlp: Linear(inner -> 4 inner), Swish, Linear(4 inner -> inner)
  const std::string mlp = c->cfg.model == FDSR_MODEL_SR3 ? "denoise_fn.time_mlp" : "denoise_fn.noise_level_mlp";
  if ((rc = need(mlp + ".1.weight", 4 * inner * inner, "embedding MLP"))) return rc;
  if ((rc = need(mlp + ".1.bias", 4 * inner, "embedding MLP"))) return rc;
  if ((rc = need(mlp + ".3.weight", 4 * inner * inner, "embedding MLP"))) return rc;
  if ((rc = need(mlp + ".3.bias", inner, "embedding MLP"))) return rc;
  for (const HAttn& a : c->attns) {
    if (a.kind != 0) continue;  // CLAM: Conv2d(C, C/16, 1), Conv2d(C/16, C, 1); SLAM: Conv2d(2, 1, 7) — all bias-free
    const std::string q = "denoise_fn." + a.name;
    const size_t C = size_t(a.C), R = C / 16;
    if ((rc = need(q + ".ca.fc1.weight", R * C, "CLAM fc1"))) return rc;
    if ((rc = need(q + ".ca.fc2.weight", C * R, "CLAM fc2"))) return rc;
    if ((rc = need(q + ".sa.conv1.weight", 98, "SLAM conv"))) return rc;
  }
  return FDSR_OK;
}

const std::vector<float>* find_w(fdsr_ctx* c, const std::string& name) {
  if (name == "@identity") {  // 256 x 256 identity (1x1 "weights" of an identity-residual K chunk)
    static const std::vector<float> eye = [] {
      std::vector<float> e(256 * 256, 0.f);
      for (int i = 0; i < 256; ++i) e[i * 256 + i] = 1.f;
      return e;
    }();
    return &eye;
  }
  auto it = c->host_w.find(name);
  return it == c->host_w.end() ? nullptr : &it->second;
}

template <typename T>
T to_t(float f);
template <>
__half to_t<__half>(float f) { return __float2half_rn(f); }
template <>
__nv_bfloat16 to_t<__nv_bfloat16>(float f) { return __float2bfloat16_rn(f); }
// weight of a chunk whose A operand is a GroupNorm output: always fp16 (GnOperand, conv_kernel.cuh); raw chunks: T
template <typename T>
T to_w(float f, bool gn_chunk) {
  if (!gn_chunk) return to_t<T>(f);
  const __half h = __float2half_rn(f);
  T r;
  static_assert(sizeof(T) == sizeof(__half), "16-bit storage");
  memcpy(&r, &h, sizeof r);
  return r;
}

template <typename T>
int pack_weights(fdsr_ctx* c) {
  // blob layout per (chunk, tap): [channel group][n][8 channels] of T  (K-major, no swizzle)
  // Pair-capable layers are packed twice: the full-width layout (single-CTA launches, split-N halves) and, at w_off2,
  // two half-width copies of the same layout — columns [0, N/2) then [N/2, N) — for CTA-pair launches.
  size_t total = 0;
  for (HConv& k : c->convs) {
    k.w_off = total;
    k.w_bytes = 0;
    for (const HChunk& ch : k.chunks) k.w_bytes += size_t(k.phases) * ch.taps.size() * size_t(k.ncg) * k.N * 16;
    total += k.w_bytes;
  }
  for (HConv& k : c->convs) {
    k.w_off2 = total;
    if (k.pair_ok()) total += k.w_bytes;
  }
  std::vector<T> host(total / sizeof(T), to_t<T>(0.f));
  for (HConv& k : c->convs) {
    size_t off = k.w_off;
    for (int ph = 0; ph < k.phases; ++ph)
    for (const HChunk& ch : k.chunks) {
      const std::vector<float>* w = find_w(c, ch.wname);
      if (!w) return fail(c, FDSR_E_NOTFOUND, "missing weight %s", ch.wname.c_str());
      const WeightGeom g(k, ch, w->size());
      for (const HTap& tp : ch.taps) {
        T* blob = host.data() + off / sizeof(T);
        for (int cg = 0; cg < k.ncg; ++cg)
          for (int n = 0; n < k.cout; ++n)
            for (int j = 0; j < 8; ++j) {
              const int wci = ch.wchan(cg * 8 + j);
              if (wci < 0) continue;
              if (k.phases == 4) {
                // tap (ry, rx) of phase (py, px): the 3x3 taps whose upsampled source row / column is that one
                const int py = ph >> 1, px = ph & 1;
                float acc = 0.f;
                for (int dy = 0; dy < 3; ++dy)
                  for (int dx = 0; dx < 3; ++dx)
                    if (((py + dy + 1) >> 1) - py == tp.ky && ((px + dx + 1) >> 1) - px == tp.kx)
                      acc += (*w)[g.at(k.w_n0 + n, wci, dy, dx)];
                blob[(size_t(cg) * k.N + n) * 8 + j] = to_w<T>(acc, ch.gn != 0);
                continue;
              }
              blob[(size_t(cg) * k.N + n) * 8 + j] = to_w<T>((*w)[g.at(k.w_n0 + n, wci, tp.ky, tp.kx)], ch.gn != 0);
            }
        off += size_t(k.ncg) * k.N * 16;
      }
    }
    if (k.pair_ok()) {  // half-width copies: element (blob, cg, n, j) -> half n / (N/2), same blob, (cg, n % (N/2), j)
      const size_t blob_e = size_t(k.ncg) * k.N * 8, nblobs = k.w_bytes / (blob_e * sizeof(T));
      const int nh = k.N / 2;
      const T* src = host.data() + k.w_off / sizeof(T);
      T* dst = host.data() + k.w_off2 / sizeof(T);
      for (size_t bi = 0; bi < nblobs; ++bi)
        for (int cg = 0; cg < k.ncg; ++cg)
          for (int n = 0; n < k.N; ++n)
            memcpy(dst + size_t(n / nh) * (nblobs * blob_e / 2) + bi * (blob_e / 2) + (size_t(cg) * nh + n % nh) * 8,
                   src + bi * blob_e + (size_t(cg) * k.N + n) * 8, 8 * sizeof(T));
    }
  }
  return upload(c, c->d_weights, host);
}

// fp32 parity mode: per conv, per chunk: [tap][ci < creal][N] floats
int pack_weights_f32(fdsr_ctx* c) {
  size_t total = 0;
  c->w32_off.assign(c->convs.size(), 0);
  for (size_t i = 0; i < c->convs.size(); ++i) {
    c->w32_off[i] = total;
    for (const HChunk& ch : c->convs[i].chunks) total += ch.taps.size() * size_t(ch.creal) * c->convs[i].N;
  }
  std::vector<float> host(total, 0.f);
  for (size_t i = 0; i < c->convs.size(); ++i) {
    const HConv& k = c->convs[i];
    size_t off = c->w32_off[i];
    for (const HChunk& ch : k.chunks) {
      const std::vector<float>* w = find_w(c, ch.wname);
      if (!w) return fail(c, FDSR_E_NOTFOUND, "missing weight %s", ch.wname.c_str());
      const WeightGeom g(k, ch, w->size());
      for (const HTap& tp : ch.taps) {
        for (int ci = 0; ci < ch.creal; ++ci) {
          const int wci = ch.wchan(ci);
          if (wci < 0) continue;
          for (int n = 0; n < k.cout; ++n)
            host[off + size_t(ci) * k.N + n] = (*w)[g.at(k.w_n0 + n, wci, tp.ky, tp.kx)];
        }
        off += size_t(ch.creal) * k.N;
      }
    }
  }
  return upload(c, c->d_weights32, host, 16);
}

int upload_params(fdsr_ctx* c) {
  std::vector<float> p;
  for (HConv& k : c->convs) {
    if (k.gn_C == 0) continue;
    const std::vector<float>*ga = find_w(c, k.gn_name + ".weight"), *be = find_w(c, k.gn_name + ".bias");
    if (!ga || !be || int(ga->size()) != k.gn_C)
      return fail(c, FDSR_E_NOTFOUND, "missing/invalid GroupNorm params %s", k.gn_name.c_str());
    k.gamma_off = p.size();
    p.insert(p.end(), ga->begin(), ga->end());
    p.insert(p.end(), be->begin(), be->end());
  }
  for (HAttn& a : c->attns) {
    if (a.kind != 0) continue;
    const std::string q = "denoise_fn." + a.name;
    const std::vector<float>*w1 = find_w(c, q + ".ca.fc1.weight"), *w2 = find_w(c, q + ".ca.fc2.weight"),
                            *w7 = find_w(c, q + ".sa.conv1.weight");
    if (!w1 || !w2 || !w7 || w7->size() != 98) return fail(c, FDSR_E_NOTFOUND, "missing CLAM/SLAM weights of %s", q.c_str());
    a.w1_off = p.size();
    p.insert(p.end(), w1->begin(), w1->end());
    a.w2_off = p.size();
    p.insert(p.end(), w2->begin(), w2->end());
    a.w7_off = p.size();
    p.insert(p.end(), w7->begin(), w7->end());
  }
  return upload(c, c->d_params, p, 16);
}

// y[o] = b[o] + sum_i w[o][i] x[i]   (fp32, like nn.Linear)
std::vector<float> linear(const std::vector<float>& w, const std::vector<float>& b, const std::vector<float>& x) {
  const size_t in = x.size(), out = b.size();
  std::vector<float> y(out);
  for (size_t o = 0; o < out; ++o) {
    float a = 0.f;
    for (size_t i = 0; i < in; ++i) a += w[o * in + i] * x[i];
    y[o] = a + b[o];
  }
  return y;
}

// Per-step bias tables: conv bias (+ res_conv bias) + FiLM(noise_level_t) (unet.py:22-54, 242-248)
int build_bias_tables(fdsr_ctx* c) {
  const int T = c->T, inner = c->cfg.inner_channel;
  const bool sr3 = c->cfg.model == FDSR_MODEL_SR3;
  // FastDiffSR embeds the noise level sqrt_alphas_cumprod_prev[t+1] (noise_level_mlp); the SR3 baseline embeds the
  // integer step t itself (time_mlp, ddpm_modules/unet.py:19-33, 165-171; diffusion.py:178)
  const std::string mlp = sr3 ? "denoise_fn.time_mlp" : "denoise_fn.noise_level_mlp";
  const auto *w1 = find_w(c, mlp + ".1.weight"), *b1 = find_w(c, mlp + ".1.bias"), *w3 = find_w(c, mlp + ".3.weight"),
             *b3 = find_w(c, mlp + ".3.bias");
  if (!w1 || !b1 || !w3 || !b3) return fail(c, FDSR_E_NOTFOUND, "missing %s weights", mlp.c_str());
  const std::vector<double>& nl = c->tables["sqrt_alphas_cumprod_prev"];
  const int count = inner / 2;
  std::vector<float> inv_freq(count);
  if (sr3) {
    const auto* fr = find_w(c, "denoise_fn.time_mlp.0.inv_freq");  // registered buffer: part of the state_dict
    for (int i = 0; i < count; ++i)
      inv_freq[i] = (fr && int(fr->size()) == count) ? (*fr)[i] : expf(float(2 * i) * (-logf(10000.f) / float(inner)));
  }
  std::vector<std::vector<float>> temb(T);
  for (int t = 0; t < T; ++t) {
    std::vector<float> enc(inner);
    if (sr3) {
      for (int i = 0; i < count; ++i) {
        const float e = float(t) * inv_freq[i];
        enc[i] = sinf(e);
        enc[count + i] = cosf(e);
      }
    } else {
      const float level = float(nl[t + 1]);
      for (int i = 0; i < count; ++i) {
        const float step = float(i) / float(count);
        const float e = level * expf(-logf(1e4f) * step);
        enc[i] = sinf(e);
        enc[count + i] = cosf(e);
      }
    }
    std::vector<float> h = linear(*w1, *b1, enc);
    for (float& v : h) v = v / (1.0f + expf(-v));
    temb[t] = linear(*w3, *b3, h);
  }
  std::vector<std::vector<float>> temb_sw = temb;  // swish(emb): input of the SR3 per-block Linear
  for (auto& e : temb_sw)
    for (float& v : e) v = v / (1.0f + expf(-v));
  size_t total = 0;
  for (HConv& k : c->convs) {
    k.bias_off = total;
    total += size_t(T) * k.N;
  }
  std::vector<float> tab(total, 0.f);
  for (HConv& k : c->convs) {
    std::vector<float> base(k.N, 0.f);
    for (const std::string& bn : k.bias_names) {
      const auto* b = find_w(c, bn);
      if (!b || int(b->size()) != k.cout) return fail(c, FDSR_E_NOTFOUND, "missing bias %s", bn.c_str());
      for (int n = 0; n < k.cout; ++n) base[n] += (*b)[n];
    }
    const std::vector<float>*fw = nullptr, *fb = nullptr;
    if (!k.film_name.empty()) {
      fw = find_w(c, k.film_name + ".weight");
      fb = find_w(c, k.film_name + ".bias");
      if (!fw || !fb) return fail(c, FDSR_E_NOTFOUND, "missing FiLM weights %s", k.film_name.c_str());
    }
    for (int t = 0; t < T; ++t) {
      float* row = tab.data() + k.bias_off + size_t(t) * k.N;
      for (int n = 0; n < k.N; ++n) row[n] = base[n];
      if (fw) {
        const std::vector<float> f = linear(*fw, *fb, k.film_swish ? temb_sw[t] : temb[t]);
        for (int n = 0; n < k.cout; ++n) row[n] += f[n];
      }
    }
  }
  c->layers_dirty = true;
  return upload(c, c->d_bias, tab, 16);
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
constexpr size_t kOffFlags = 64;  // status word inside the fixed first 256 bytes of the workspace (after SampleArgs)

// cuTensorMapEncodeTiled through the runtime (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// A tiled TMA map of a 16-bit tensor: L2 promotion of 128 bytes, zero fill outside the tensor
constexpr cuuint32_t kUnitStrides[4] = {1, 1, 1, 1};
bool encode_map(CUtensorMap* m, const void* ptr, int rank, const cuuint64_t* dims, const cuuint64_t* strides,
                const cuuint32_t* box, const cuuint32_t* elem_strides, CUtensorMapSwizzle swizzle, bool bf16) {
  EncodeTiledFn enc = get_encode_tiled();
  return enc && enc(m, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, rank,
                    const_cast<void*>(ptr), dims, strides, box, elem_strides, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// NHWC 16-bit activation [B][H][W][C] as a rank-4 TMA tensor {C, W, H, B}, box {32, 8, 4, 1}, 64B swizzle
bool make_out_map(CUtensorMap* m, void* ptr, int B, int H, int W, int C, bool bf16) {
  const cuuint64_t dims[4] = {cuuint64_t(C), cuuint64_t(W), cuuint64_t(H), cuuint64_t(B)};
  const cuuint64_t strides[3] = {cuuint64_t(C) * 2, cuuint64_t(W) * C * 2, cuuint64_t(H) * W * C * 2};
  const cuuint32_t box[4] = {32, cuuint32_t(kTileW), 4, 1};
  return encode_map(m, ptr, 4, dims, strides, box, kUnitStrides, CU_TENSOR_MAP_SWIZZLE_64B, bf16);
}

// Output of a phase-decomposed upsample conv: parity (py, px) = (ph >> 1, ph & 1) of the NHWC 16-bit tensor
// [B][2h][2w][C] viewed as a rank-4 tensor {C, w, h, B} over the low-resolution grid
bool make_out_map_phase(CUtensorMap* m, void* ptr, int B, int h, int w, int C, int ph, bool bf16) {
  const int Wo = 2 * w, Ho = 2 * h;
  uint8_t* base = static_cast<uint8_t*>(ptr) + (size_t(ph >> 1) * Wo + (ph & 1)) * C * 2;
  const cuuint64_t dims[4] = {cuuint64_t(C), cuuint64_t(w), cuuint64_t(h), cuuint64_t(B)};
  const cuuint64_t strides[3] = {cuuint64_t(C) * 4, cuuint64_t(Wo) * C * 4, cuuint64_t(Ho) * Wo * C * 2};
  const cuuint32_t box[4] = {32, cuuint32_t(kTileW), 4, 1};
  return encode_map(m, base, 4, dims, strides, box, kUnitStrides, CU_TENSOR_MAP_SWIZZLE_64B, bf16);
}

// NHWC 16-bit source [B][H][W][C] as a rank-4 TMA tensor {C, W, H, B}, box {64 ch, 10, 34, 1}, 128B swizzle:
// one load = one 64-channel input patch with halo, pixel-major 128-byte rows, zero-filled outside the image
// kind 0: full patch; 1: centre box {64, 8, 32}; 2: space-to-depth plane = box {64, 20, 68} traversed with element
// strides {1, 2, 2, 1} (every second pixel in x and y: 10 x 34 positions land in shared memory)
bool make_in_map(CUtensorMap* m, const void* ptr, int B, int H, int W, int C, bool bf16, int kind, int tile_h = kTileH) {
  const cuuint64_t dims[4] = {cuuint64_t(C), cuuint64_t(W), cuuint64_t(H), cuuint64_t(B)};
  const cuuint64_t strides[3] = {cuuint64_t(C) * 2, cuuint64_t(W) * C * 2, cuuint64_t(H) * W * C * 2};
  if (kind == 3) {  // 16-channel stem input: one 8-channel plane of the patch per load (box {8, 10, 34}), no swizzle
    const cuuint32_t box[4] = {8, cuuint32_t(kPatchW), cuuint32_t(kPatchH), 1};
    return C == 16 && encode_map(m, ptr, 4, dims, strides, box, kUnitStrides, CU_TENSOR_MAP_SWIZZLE_NONE, bf16);
  }
  const cuuint32_t sc = kind == 2 ? 2 : 1;
  const cuuint32_t box[4] = {64, cuuint32_t(kind == 1 ? kTileW : kPatchW) * sc, cuuint32_t(kind == 1 ? tile_h : tile_h + 2) * sc, 1};
  const cuuint32_t estr[4] = {1, sc, sc, 1};
  return C >= 64 && encode_map(m, ptr, 4, dims, strides, box, estr, CU_TENSOR_MAP_SWIZZLE_128B, bf16);
}

// [B][HW][C] 16-bit token matrix (an NHWC activation seen as rows of C channels) as a rank-3 TMA tensor
// {C, HW, B}, box {64 ch, rows, 1}, 128B swizzle: K-major (q, k) / MN-major (v) MMA operand tiles
bool make_token_map(CUtensorMap* m, const void* ptr, int B, int HW, int C, int rows, bool bf16) {
  const cuuint64_t dims[3] = {cuuint64_t(C), cuuint64_t(HW), cuuint64_t(B)};
  const cuuint64_t strides[2] = {cuuint64_t(C) * 2, cuuint64_t(HW) * C * 2};
  const cuuint32_t box[3] = {64, cuuint32_t(rows), 1};
  return encode_map(m, ptr, 3, dims, strides, box, kUnitStrides, CU_TENSOR_MAP_SWIZZLE_128B, bf16);
}

// SelfAttention cores of the SR3 baseline (16-bit modes): tensor maps of q / k / v at the reserved shape
int upload_attn(fdsr_ctx* c) {
  c->a_params.assign(c->attns.size(), AttnParams{});
  const bool bf = c->cfg.dtype == FDSR_DTYPE_BF16;
  for (size_t i = 0; i < c->attns.size(); ++i) {
    const HAttn& a = c->attns[i];
    if (a.kind != 1 || c->attn_ref) continue;
    const HTensor& tq = c->tensors[a.tq];
    const int HW = (c->H >> tq.level) * (c->W >> tq.level);
    AttnParams& p = c->a_params[i];
    if (!make_token_map(&p.q_map, c->d_ws + tq.off, c->B, HW, a.C, kAttnQ, bf) ||
        !make_token_map(&p.k_map, c->d_ws + c->tensors[a.tk].off, c->B, HW, a.C, kAttnKB, bf) ||
        !make_token_map(&p.v_map, c->d_ws + c->tensors[a.tv].off, c->B, HW, a.C, kAttnKB, bf))
      return fail(c, FDSR_E_CUDA, "cuTensorMapEncodeTiled failed for the attention operands of %s", a.name.c_str());
    p.out = c->d_ws + c->tensors[a.out].off;
    p.HW = HW;
    p.scale_log2 = 1.4426950408889634f / sqrtf(float(a.C));
  }
  return FDSR_OK;
}

// fp32 parity mode: layer descriptions for conv_f32_kernel / f32_gn_table_kernel
int upload_layers_f32(fdsr_ctx* c) {
  const int B = c->B, H = c->H, W = c->W;
  c->f_layers.assign(c->convs.size(), F32Layer{});
  c->f_gn.assign(c->convs.size(), F32GnArgs{});
  for (size_t i = 0; i < c->convs.size(); ++i) {
    const HConv& k = c->convs[i];
    F32Layer& l = c->f_layers[i];
    memset(&l, 0, sizeof l);
    const int lvl = k.out >= 0 ? c->tensors[k.out].level : 0;
    l.B = B;
    l.H = H >> lvl;
    l.W = W >> lvl;
    l.N = k.N;
    l.mode = k.mode;
    l.nchunks = int(k.chunks.size());
    size_t woff = c->w32_off[i];
    for (int j = 0; j < l.nchunks; ++j) {
      const HChunk& ch = k.chunks[j];
      const HTensor& t = c->tensors[k.src[ch.slot]];
      F32Chunk& d = l.chunk[j];
      d.src = reinterpret_cast<const float*>(c->d_ws + t.off);
      d.C = t.C;
      d.H = H >> t.level;
      d.W = W >> t.level;
      d.c0 = ch.c0;
      d.nch = ch.creal;
      d.gn = ch.gn;
      d.vc0 = ch.vc0;
      d.pa = ch.parity < 0 ? 0 : (ch.parity >> 1);
      d.pb = ch.parity < 0 ? 0 : (ch.parity & 1);
      d.ntaps = int(ch.taps.size());
      for (int tp = 0; tp < d.ntaps; ++tp) {
        d.dy[tp] = int8_t(ch.taps[tp].pos / kPatchW - 1);
        d.dx[tp] = int8_t(ch.taps[tp].pos % kPatchW - 1);
      }
      d.w_off = int32_t(woff - c->w32_off[i]);
      woff += ch.taps.size() * size_t(ch.creal) * k.N;
    }
    l.gn_C = k.gn_C;
    l.gn_tab = reinterpret_cast<const float2*>(c->d_ws + c->off_gntab);
    l.weights = c->d_weights32 + c->w32_off[i];
    l.bias = c->d_bias + k.bias_off;
    l.bias_tstride = k.N;
    l.resid = k.resid >= 0 ? reinterpret_cast<const float*>(c->d_ws + c->tensors[k.resid].off) : nullptr;
    l.out_mode = k.out_mode;
    l.out_c = k.out_c;
    if (k.out_mode == kOutAct) {
      const HTensor& t = c->tensors[k.out];
      l.out = reinterpret_cast<float*>(c->d_ws + t.off);
      l.out_stats = t.stats ? reinterpret_cast<unsigned long long*>(c->d_ws + t.stats_off) : nullptr;
      l.out_sq_scale = stat_sq_scale((long long)l.H * l.W);
    } else {
      l.out = reinterpret_cast<float*>(c->d_ws + c->off_eps);
    }
    if (k.gn_C) {
      F32GnArgs& g = c->f_gn[i];
      for (int s2 = 0; s2 < k.gn_nsrc && s2 < 2; ++s2) {
        const HTensor& t = c->tensors[k.src[s2]];
        g.stats[s2] = reinterpret_cast<const unsigned long long*>(c->d_ws + t.stats_off);
        g.C[s2] = t.C;
      }
      if (k.gn_nsrc == 1) {
        g.stats[1] = g.stats[0];
        g.C[1] = 0;
      }
      const HTensor& t0 = c->tensors[k.src[0]];
      g.gn_C = k.gn_C;
      g.groups = c->cfg.norm_groups;
      g.HW = (H >> t0.level) * (W >> t0.level);
      g.sq_scale = stat_sq_scale((long long)g.HW);
      g.eps = 1e-5f;
      g.gamma = c->d_params + k.gamma_off;
      g.beta = c->d_params + k.gamma_off + k.gn_C;
      g.tab = reinterpret_cast<float2*>(c->d_ws + c->off_gntab);
    }
  }
  static_assert(sizeof(F32Layer) <= 4000, "F32Layer must fit the kernel parameter space");
  c->layers_dirty = false;
  return FDSR_OK;
}

int launch_conv_f32(fdsr_ctx* c, int li, int t, cudaStream_t st) {
  const HConv& k = c->convs[li];
  const F32Layer& l = c->f_layers[li];
  if (k.gn_C) {
    const int rc = launch(c, f32_gn_table_kernel, c->B, 256, 0, st, c->f_gn[li]);
    if (rc) return rc;
  }
  const int tiles = c->B * ((l.W + kF32Tile - 1) / kF32Tile) * ((l.H + kF32Tile - 1) / kF32Tile);
  return launch(c, conv_f32_kernel, dim3(tiles, (l.N + kF32NBlk - 1) / kF32NBlk), 256, 0, st, l, t);
}

int upload_layers(fdsr_ctx* c) {
  if (c->cfg.dtype == FDSR_DTYPE_FP32) return upload_layers_f32(c);
  const int B = c->B, H = c->H, W = c->W;
  const bool bf = c->cfg.dtype == FDSR_DTYPE_BF16;
  if (!c->d_prof) {
    CUDA_TRY(c, c->d_prof.grow(size_t(c->num_sms) * kProfRoles * 64));
    CUDA_TRY(c, cudaMemset(c->d_prof, 0, size_t(c->num_sms) * kProfRoles * 64));
  }
  std::vector<ConvLayer> L(c->convs.size());
  for (size_t i = 0; i < c->convs.size(); ++i) {
    const HConv& k = c->convs[i];
    ConvLayer& l = L[i];
    memset(&l, 0, sizeof l);
    const int lvl = k.out >= 0 ? c->tensors[k.out].level : 0;
    l.B = B;
    l.phases = k.phases;
    // a phase layer tiles the low-resolution grid once per output parity (virtual images = B * 4)
    l.H = (H >> lvl) >> (k.phases == 4 ? 1 : 0);
    l.W = (W >> lvl) >> (k.phases == 4 ? 1 : 0);
    l.tiles_x = (l.W + kTileW - 1) / kTileW;
    // Half tiles (16 x 8 pixels, one MMA tile per CTA tile), run as CTA pairs, for the wide layers whose 32 x 8 tiles
    // would not fill the GPU (32^2 at B = 16: 64 tiles; everything below 256^2 at B = 1): twice the CTAs, half the patch
    // each CTA loads and normalises, and N = 256 gets a second TMEM accumulator stage.  The weight bytes per pixel double,
    // which is why layers with enough full tiles keep them (64^2 at B = 16: measured 1.3 % slower per step as half tiles).
    // Results are bit-identical for either shape (per-warp statistics are added as integers), so the choice may follow B.
    const int full_tiles = B * l.tiles_x * ((l.H + kTileH - 1) / kTileH);
    const bool half = c->half_tiles && c->pair && k.mode == kModeNormal && k.ncg == 8 && k.phases == 1 &&
                      k.out_mode == kOutAct && k.N >= 128 && l.tiles_x % 2 == 0 && l.H % 16 == 0 && full_tiles <= c->num_sms;
    l.tile_h = half ? 16 : kTileH;
    l.tiles_y = (l.H + l.tile_h - 1) / l.tile_h;
    l.ntiles = B * k.phases * l.tiles_x * l.tiles_y;
    // Split-N: a low-resolution layer with fewer 256-pixel tiles than half the SMs is computed as two
    // 128-column halves by twice as many CTAs.  Only 256 -> 2 x 128: both widths use the same
    // per-tile statistics path, so results stay bitwise independent of the batch size.
    l.nsplit = (!half && c->split_n && k.out_mode == kOutAct && k.N == 256 && 2 * l.ntiles <= c->num_sms) ? 2 : 1;
    l.n_full = k.N;
    l.N = k.N / l.nsplit;
    l.ncg = k.ncg;
    l.mode = k.mode;
    for (int s = 0; s < k.nsrc; ++s) {
      const HTensor& t = c->tensors[k.src[s]];
      l.src[s].ptr = c->d_ws + t.off;
      l.src[s].stats = t.stats ? reinterpret_cast<const unsigned long long*>(c->d_ws + t.stats_off) : nullptr;
      l.src[s].C = t.C;
      l.src[s].H = H >> t.level;
      l.src[s].W = W >> t.level;
    }
    // Input patches arrive by TMA, except in the nine-tap upsample convs, whose producer warps gather the 2x patch.
    // The stem's 16-channel input arrives as two 8-channel plane loads (no producer work).
    l.a_tma = k.mode == kModeUp2x ? 0 : (k.ncg == 2 ? 2 : 1);
    bool maps_ok = l.a_tma != 2 || make_in_map(&l.in_map[0], l.src[0].ptr, B, l.src[0].H, l.src[0].W, l.src[0].C, bf, 3);
    for (int s = 0; s < k.nsrc && l.a_tma == 1; ++s)
      maps_ok = maps_ok &&
                make_in_map(&l.in_map[s], l.src[s].ptr, B, l.src[s].H, l.src[s].W, l.src[s].C, bf, 0, l.tile_h) &&
                make_in_map(&l.in_map_c[s], l.src[s].ptr, B, l.src[s].H, l.src[s].W, l.src[s].C, bf,
                            k.mode == kModeS2D ? 2 : 1, l.tile_h);
    if (!maps_ok) return fail(c, FDSR_E_CUDA, "layer %s: tensor maps of the input patches failed", k.name.c_str());
    l.nchunks = int(k.chunks.size());
    int any_center = 0;
    size_t woff = 0;
    for (int j = 0; j < l.nchunks; ++j) {
      const HChunk& ch = k.chunks[j];
      ConvChunk& d = l.chunk[j];
      d.src = ch.slot;
      d.c0 = ch.c0;
      d.gn = ch.gn;
      d.vc0 = ch.vc0;
      d.ntaps = int(ch.taps.size());
      d.w_off = int(woff);
      for (int tp = 0; tp < d.ntaps; ++tp) d.tap_pos[tp] = ch.taps[tp].pos;
      d.parity = ch.parity < 0 ? 0 : ch.parity;
      d.center = (k.mode == kModeNormal && ch.gn == 0 && d.ntaps == 1 && d.tap_pos[0] == kPatchW + 1) ? 1 : 0;
      any_center += d.center;
      woff += ch.taps.size() * size_t(k.ncg) * k.N * 16;
    }
    // patch rings (see ConvCfg): N = 64 layers with 1x1-residual chunks use 2 full + 2 centre-box stages
    // (with three centre boxes per tile two 32 KB stages stall on the third: measured slower in both rounds,
    //  ups.12.block2 189.6 -> 200.9 us as CTA pairs, profiles/r2/epilogue_costs.log)
    l.nR = (any_center >= 1 && any_center <= 2 && l.N == 64) ? 2 : 0;
    l.nG = l.nR ? 2 : (l.N >= 256 ? 2 : 3);
    for (int j = 0; j < l.nchunks; ++j) l.chunk[j].ring = (l.nR && l.chunk[j].center) ? 1 : 0;
    l.gn_C = k.gn_C;
    l.gn_nsrc = k.gn_nsrc;
    l.gn_groups = c->cfg.norm_groups;
    l.gn_eps = 1e-5f;
    if (k.gn_C) {
      l.gamma = c->d_params + k.gamma_off;
      l.beta = c->d_params + k.gamma_off + k.gn_C;
      const double hw = double(l.src[0].H) * l.src[0].W, n = double(k.gn_C / c->cfg.norm_groups) * hw;
      l.gn_inv_sum = 1.0 / (kStatScale * n);
      l.gn_inv_sq = 1.0 / (stat_sq_scale((long long)hw) * n);
    }
    l.bias = c->d_bias + k.bias_off;
    l.bias_tstride = k.N;
    l.resid = k.resid >= 0 ? c->d_ws + c->tensors[k.resid].off : nullptr;
    l.out_mode = k.out_mode;
    l.out_c = k.out_c;
    if (k.out_mode == kOutAct) {
      const HTensor& t = c->tensors[k.out];
      l.out = c->d_ws + t.off;
      bool ok = true;  // (the epilogue stores N >= 32 activations by TMA)
      if (k.phases == 4)
        for (int ph = 0; ph < 4 && ok; ++ph)
          ok = make_out_map_phase(ph == 0 ? &l.out_map : &l.out_map_ph[ph - 1], l.out, B, l.H, l.W, k.N, ph, bf);
      else if (k.N >= 32)
        ok = make_out_map(&l.out_map, l.out, B, l.H, l.W, k.N, bf);
      if (!ok) return fail(c, FDSR_E_CUDA, "layer %s: tensor maps of the output failed", k.name.c_str());
      l.out_stats = t.stats ? reinterpret_cast<unsigned long long*>(c->d_ws + t.stats_off) : nullptr;
      l.out_sq_scale = float(stat_sq_scale((long long)(H >> t.level) * (W >> t.level)));
      int su = 1;
      while (su < 8 && t.unit % (4 * su) == 0) su *= 2;  // largest power of two with 2*su | unit, <= 8 pairs
      l.out_su = (l.N == 64) ? 1 : su;                    // N = 64 keeps per-pair running sums in TMEM
    } else {
      l.out = c->d_ws + c->off_eps;
    }
    // CTA pairs (cta_group::2): TMA-fed layers whose tile rows have an even number of tiles (a pair = two x-neighbours);
    // the choice depends on the layer and the image shape only, never on B, so results do not depend on the batch size
    l.pair = (c->pair && k.pair_ok() && l.a_tma && l.nsplit == 1 && l.tiles_x % 2 == 0) ? 1 : 0;
    l.weights = c->d_weights + (l.pair ? k.w_off2 : k.w_off);
    l.w_half = int32_t(k.w_bytes / 2);
    {
      const int tpi = l.tiles_x * l.tiles_y;
      // running TMEM statistics exist for N = 64 only; the group size must not depend on B.  A CTA's consecutive tiles
      // are t, t+1 (single) or t, t+2 (pair): both of a group must belong to one image
      l.group = (l.N == 64 && tpi % (l.pair ? 4 : 2) == 0) ? 2 : 1;
    }
    {  // second epilogue team (warps 12..19) for layers whose producer warps have nothing to do
      // (not the stride-2 convs: they stream four parity-plane chunks per tile and lose more from giving up the third
      //  patch stage than they gain — measured 49.6 -> 58.8 us for downs.3)
      bool raw = k.mode == kModeNormal && k.out_mode == kOutAct && l.tile_h == kTileH && l.nsplit == 1 && k.resid < 0;
      for (const HChunk& ch : k.chunks) raw = raw && ch.gn == 0;
      l.epi2 = (c->epi2 && raw) ? 1 : 0;
      if (l.epi2 && l.N <= 128) {  // their staging blocks live in the third patch stage
        l.nG = 2;
        l.nR = 0;
        for (int j = 0; j < l.nchunks; ++j) l.chunk[j].ring = 0;
      }
    }
    l.tail2 = (c->tail_help && !l.epi2 && k.out_mode == kOutAct && l.N >= 64) ? 1 : 0;
    l.prof = c->d_prof;
    l.flags = reinterpret_cast<unsigned int*>(c->d_ws + kOffFlags);
  }
  static_assert(sizeof(ConvLayer) <= 4000, "ConvLayer must fit the kernel parameter space");
  // the sampler's form of the final conv: eps stays in registers, the epilogue performs the posterior update
  c->final_fused = L.back();
  c->final_fused.out_mode = kOutPosterior;
  c->final_fused.post = c->d_post;
  c->final_fused.x_state = reinterpret_cast<float*>(c->d_ws + c->off_x);
  c->final_fused.xin = c->d_ws + c->tensors[c->t_xin].off;
  c->final_fused.args = reinterpret_cast<const SampleArgs*>(c->d_ws + c->off_seed);
  c->h_layers = L;
  const int rc = upload_attn(c);
  if (rc) return rc;
  c->layers_dirty = false;
  return FDSR_OK;
}

// The launch descriptors point into the workspace and the weight, parameter, bias and posterior buffers: rebuilt after
// any of them moved or changed shape
int ensure_layers(fdsr_ctx* c) { return c->layers_dirty ? upload_layers(c) : FDSR_OK; }

template <int N, typename T>
cudaError_t set_conv_attr() {
  cudaError_t e = cudaFuncSetAttribute(conv_gemm_kernel<N, T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       ConvCfg<N>::kSmemBytes);
  if constexpr (N >= 64) {
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(conv_gemm_kernel<N, T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               ConvCfg<N>::kSmemBytes);
  }
  return e;
}
template <typename T>
cudaError_t set_conv_attrs() {
  cudaError_t e = set_conv_attr<16, T>();
  if (e == cudaSuccess) e = set_conv_attr<64, T>();
  if (e == cudaSuccess) e = set_conv_attr<128, T>();
  if (e == cudaSuccess) e = set_conv_attr<256, T>();
  return e;
}

template <typename T>
int launch_conv16(fdsr_ctx* c, int li, int t, cudaStream_t st, const ConvLayer* override_layer = nullptr);

// CTAs of one conv launch (the kernel divides the layer's tile groups evenly over them, see conv_gemm_kernel)
int conv_grid(const fdsr_ctx* c, const ConvLayer& l) {
  const int cs = l.pair ? 2 : 1;  // CTA pairs are clusters of two; the unit of work is then a pair of tiles
  const int ngroups = l.ntiles / cs / l.group;
  int grid = (ngroups < c->num_sms / cs ? ngroups : c->num_sms / cs) * cs;
  if (l.nsplit > 1) {  // nsplit CTAs per tile group; persistent over the groups when there are more than fit one wave
    grid = ngroups * l.nsplit;
    if (grid > c->num_sms) grid = c->num_sms - c->num_sms % l.nsplit;
  }
  return grid;
}

template <int N, typename T>
int launch_conv_t(fdsr_ctx* c, int li, int t, cudaStream_t st, const ConvLayer* override_layer) {
  const ConvLayer& LY = override_layer ? *override_layer : c->h_layers[li];
  const bool pair = c->h_layers[li].pair != 0;
  const int cs = pair ? 2 : 1;
  const int grid = conv_grid(c, c->h_layers[li]);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kConvThreads);
  cfg.dynamicSmemBytes = ConvCfg<N>::kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cs;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  void (*kernel)(ConvLayer, int) = conv_gemm_kernel<N, T, false>;
  if constexpr (N >= 64) {
    if (pair) kernel = conv_gemm_kernel<N, T, true>;
  }
  return launched(c, cudaLaunchKernelEx(&cfg, kernel, LY, t), reinterpret_cast<const void*>(kernel));
}

template <typename T>
int launch_conv(fdsr_ctx* c, int li, int t, cudaStream_t st, const ConvLayer* override_layer = nullptr) {
  if constexpr (sizeof(T) == 4) return launch_conv_f32(c, li, t, st);
  else return launch_conv16<T>(c, li, t, st, override_layer);
}

template <typename T>
int launch_conv16(fdsr_ctx* c, int li, int t, cudaStream_t st, const ConvLayer* override_layer) {
  const HConv& k = c->convs[li];
  switch (c->h_layers[li].N) {
    case 16: return launch_conv_t<16, T>(c, li, t, st, override_layer);
    case 64: return launch_conv_t<64, T>(c, li, t, st, override_layer);
    case 128: return launch_conv_t<128, T>(c, li, t, st, override_layer);
    case 256: return launch_conv_t<256, T>(c, li, t, st, override_layer);
  }
  return fail(c, FDSR_E_INVALID, "unsupported N=%d", k.N);
}

// The tensor-core SelfAttention core for C channels (64, 128 or 256) and its dynamic shared memory
template <typename T>
std::pair<void (*)(AttnParams), int> attn_core(int C) {
  if (C == 64) return {attn_core_kernel<T, 64>, AttnCfg<64>::kSmemBytes};
  if (C == 128) return {attn_core_kernel<T, 128>, AttnCfg<128>::kSmemBytes};
  if (C == 256) return {attn_core_kernel<T, 256>, AttnCfg<256>::kSmemBytes};
  return {nullptr, 0};
}

template <typename T>
int launch_self_attn(fdsr_ctx* c, int ai, cudaStream_t st) {
  const HAttn& a = c->attns[ai];
  const HTensor& tq = c->tensors[a.tq];
  const int HW = (c->H >> tq.level) * (c->W >> tq.level), C = a.C;
  if constexpr (sizeof(T) == 2) {
    if (!c->attn_ref) {
      const auto core = attn_core<T>(C);
      if (!core.first) return fail(c, FDSR_E_INVALID, "SelfAttention with %d channels", C);
      return launch(c, core.first, dim3((HW + kAttnQ - 1) / kAttnQ, c->B), kAttnQ, core.second, st, c->a_params[ai]);
    }
  }
  return launch(c, attn_core_ref_kernel<T>, dim3((HW + 7) / 8, c->B), 256, 0, st,
                reinterpret_cast<const T*>(c->d_ws + tq.off), reinterpret_cast<const T*>(c->d_ws + c->tensors[a.tk].off),
                reinterpret_cast<const T*>(c->d_ws + c->tensors[a.tv].off),
                reinterpret_cast<T*>(c->d_ws + c->tensors[a.out].off), HW, C, 1.0f / sqrtf(float(C)));
}

template <typename T>
int launch_attn(fdsr_ctx* c, int ai, cudaStream_t st) {
  const HAttn& a = c->attns[ai];
  if (a.kind == 1) return launch_self_attn<T>(c, ai, st);
  const HTensor& ti = c->tensors[a.in];
  const HTensor& to = c->tensors[a.out];
  const int h = c->H >> ti.level, w = c->W >> ti.level, HW = h * w, C = a.C, R = C / 16;
  const T* x = reinterpret_cast<const T*>(c->d_ws + ti.off);
  T* y = reinterpret_cast<T*>(c->d_ws + to.off);
  unsigned long long* psum = reinterpret_cast<unsigned long long*>(c->d_ws + c->off_psum);
  uint32_t* pmax = reinterpret_cast<uint32_t*>(c->d_ws + c->off_pmax);
  float* gate = reinterpret_cast<float*>(c->d_ws + c->off_gate);
  float2* sp = reinterpret_cast<float2*>(c->d_ws + c->off_sp);
  const int ppb = 32;
  const int64_t nwarp = int64_t(c->B) * HW;
  int rc = launch(c, clam_pool_kernel<T>, dim3((HW + ppb - 1) / ppb, c->B), 128, 0, st, x, psum, pmax, HW, C, ppb);
  if (!rc)
    rc = launch(c, clam_gate_kernel, c->B, 256, (2 * C + 2 * R) * 4, st, psum, pmax, c->d_params + a.w1_off,
                c->d_params + a.w2_off, gate, HW, C, R);
  if (!rc) rc = launch(c, slam_pool_kernel<T>, unsigned((nwarp * 32 + 255) / 256), 256, 0, st, x, gate, sp, c->B, HW, C);
  if (!rc)
    rc = launch(c, slam_apply_kernel<T>, dim3((HW + 7) / 8, c->B), 256, 8 * C * 4, st, x, gate, sp,
                c->d_params + a.w7_off, y, reinterpret_cast<unsigned long long*>(c->d_ws + to.stats_off), h, w, C,
                stat_sq_scale((long long)h * w));
  return rc;
}

template <typename T>
int pack_input(fdsr_ctx* c, cudaStream_t st) {
  const int HW = c->H * c->W;
  const int64_t npix = int64_t(c->B) * HW;
  return launch(c, pack_input_kernel<T>, unsigned((npix + 255) / 256), 256, 0, st,
                reinterpret_cast<const float*>(c->d_ws + c->off_cond), reinterpret_cast<const float*>(c->d_ws + c->off_x),
                reinterpret_cast<T*>(c->d_ws + c->tensors[c->t_xin].off), c->B, HW, c->bands());
}

// One UNet evaluation on the context's internal cond / x buffers.
//   fused = false: cat[cond, x] is packed first and eps lands in the internal eps buffer (the fdsr_unet_forward hook);
//   fused = true (sampler): the packed input already holds x_t (written by the previous step's epilogue) and the final
//                  conv's epilogue turns eps into x_{t-1} in place (kOutPosterior) — no pack / posterior launches.
//   packed = true (tiled sampler): the network input was assembled by tile_pack_kernel; eps lands in the eps buffer.
template <typename T>
int unet_internal(fdsr_ctx* c, int t, cudaStream_t st, bool fused, bool packed = false) {
  int rc = ensure_layers(c);
  if (rc) return rc;
  CUDA_TRY(c, cudaMemsetAsync(c->d_ws + c->stats_off, 0, c->stats_bytes, st));
  if (!fused && !packed) {
    rc = pack_input<T>(c, st);
    if (rc) return rc;
  }
  for (size_t i = 0; i < c->ops.size(); ++i) {
    const HOp& op = c->ops[i];
    const bool last = fused && i + 1 == c->ops.size();
    rc = op.kind == 0 ? launch_conv<T>(c, op.idx, t, st, last ? &c->final_fused : nullptr) : launch_attn<T>(c, op.idx, st);
    if (rc) return rc;
  }
  return FDSR_OK;
}

// the fused tail exists for the 16-bit tensor-core path of the FastDiffSR model
bool can_fuse_tail(const fdsr_ctx* c) {
  return c->fused_tail && c->cfg.dtype != FDSR_DTYPE_FP32 && c->cfg.model == FDSR_MODEL_FASTDIFFSR && c->d_post.ptr != nullptr;
}

int unet_dispatch(fdsr_ctx* c, int t, cudaStream_t st, bool fused = false) {
  return with_dtype(c, [&](auto e) { return unet_internal<typename decltype(e)::type>(c, t, st, fused); });
}

int check_ready(fdsr_ctx* c) {
  if (!c->weights_loaded) return fail(c, FDSR_E_STATE, "fdsr_load_weights has not been called");
  if (c->T == 0) return fail(c, FDSR_E_STATE, "fdsr_set_schedule has not been called");
  return FDSR_OK;
}

// x_{t-1} from (x_t, eps): `images` blocks of numel_img floats.  z: explicit tensor, or (args) block z_block of the
// injected noise / the generator's stream t
int posterior_launch(fdsr_ctx* c, const float* x, const float* eps, const float* z, int t, float* out,
                     int64_t numel_img, int images, const SampleArgs* args, int64_t z_block, cudaStream_t st) {
  const int C = c->bands();
  if (numel_img % C || numel_img / C > 0x7fffffffLL || images < 1 || images > 65535)
    return fail(c, FDSR_E_INVALID, "posterior: images are (%d,H,W) blocks, 1..65535 of them", C);
  const uint32_t hw = uint32_t(numel_img / C);
  return launch(c, posterior_kernel, dim3((hw + 255) / 256, images), 256, 0, st, x, eps, z, out, hw, C, c->post[t], args,
                z_block, uint32_t(t), t > 0 ? 1 : 0);
}

// Trace frames are written after the steps t with t % trace_every(T) == 0 (and one frame before the first step)
int trace_every(int T) { return 1 | (T / 10); }

// The part of a tiled canvas one rank writes (fdsr_sample_tiled_part): the pixels whose first covering tile lies in the
// own range [g0, g1); res2img_owned_kernel writes +0.0 everywhere else
struct TileOwner {
  TileAxis ay, ax;
  int64_t g0, g1;
};

// The T-step chain of both samplers on B images of C x HW values: x_T from the generator, a trace frame before the
// first step, step(t, k) for the k-th step t = T-1 .. 0, a trace frame after every trace_every(T)-th step, and the
// result sr.  Everything that differs between two calls of the same shape (seed, image offset, noise / trace pointers)
// is read from the SampleArgs slot in device memory.  owner != nullptr: frames and result at the owner's pixels only.
template <typename Step>
int sample_chain(fdsr_ctx* c, const SampleArgs* args, float* x, const float* cond, float* sr, int B, uint32_t HW,
                 bool has_trace, cudaStream_t st, Step&& step, const TileOwner* owner = nullptr) {
  const int T = c->T, nfr = fdsr_trace_frames(c), inter = trace_every(T);
  const int64_t per = int64_t(c->bands()) * HW;
  const unsigned gb = unsigned((per * B + 255) / 256);
  // FastDiffSR predicts the residual: frames and result go through res2img (diffusion.py:213-216, 275-281).
  // The SR3 baseline predicts the image: frames are the raw x, the first frame is the conditioning image itself
  // (ddpm_modules/diffusion.py:218-227).
  const int sr3 = c->cfg.model == FDSR_MODEL_SR3 ? 1 : 0;
  const dim3 grid(unsigned((uint64_t(HW) + 255) / 256), unsigned(B));
  auto res2img = [&](const float* src, float* out, int64_t bstride, int64_t frame_off) {
    if (owner)
      return launch(c, res2img_owned_kernel, grid, 256, 0, st, src, cond, out, bstride, c->bands(), owner->ay, owner->ax,
                    owner->g0, owner->g1, args, frame_off);
    return launch(c, res2img_kernel, gb, 256, 0, st, src, cond, out, per, bstride, B, args, frame_off, sr3);
  };
  int rc = launch(c, noise_init_kernel, grid, 256, 0, st, x, HW, c->bands(), args, uint32_t(T));
  if (rc) return rc;
  int frame = 0;
  if (has_trace) {
    rc = res2img(cond, nullptr, per * nfr, 0);
    if (rc) return rc;
    frame = 1;
  }
  for (int k = 0, t = T - 1; t >= 0; --t, ++k) {
    rc = step(t, k);
    if (rc) return rc;
    if (has_trace && t % inter == 0) {
      rc = res2img(x, nullptr, per * nfr, per * frame);
      if (rc) return rc;
      ++frame;
    }
  }
  return res2img(x, sr, per, 0);
}

// The T-step loop on the context's buffers
int sample_enqueue(fdsr_ctx* c, bool has_trace, cudaStream_t st) {
  const SampleArgs* args = reinterpret_cast<const SampleArgs*>(c->d_ws + c->off_seed);
  const int64_t per = int64_t(c->bands()) * c->H * c->W;
  float* x = reinterpret_cast<float*>(c->d_ws + c->off_x);
  const float* cond = reinterpret_cast<const float*>(c->d_ws + c->off_cond);
  const float* eps = reinterpret_cast<const float*>(c->d_ws + c->off_eps);
  float* sr = reinterpret_cast<float*>(c->d_ws + c->off_sr);
  const bool fused = can_fuse_tail(c);
  return sample_chain(c, args, x, cond, sr, c->B, uint32_t(c->H) * c->W, has_trace, st, [&](int t, int k) {
    int rc = FDSR_OK;
    if (fused && k == 0) {  // cat[cond, x_T] once; afterwards every step's epilogue rewrites the x channels of the packed input
      rc = ensure_layers(c);
      if (!rc) rc = with_dtype16(c, [&](auto e) { return pack_input<typename decltype(e)::type>(c, st); });
    }
    if (!rc) rc = unet_dispatch(c, t, st, fused);
    if (!rc && !fused) rc = posterior_launch(c, x, eps, nullptr, t, x, per, c->B, args, k + 1, st);
    return rc;
  });
}

// One axis of the tile grid (the rule stated in tile_kernels.cuh / include/fdsr.h)
TileAxis make_axis(int L, int t, int overlap) {
  TileAxis a;
  a.L = L;
  a.te = std::min(t, L / 8 * 8);
  a.oe = std::min(overlap, a.te - 8);
  a.s = a.te - a.oe;
  a.n = L > a.te ? (L - a.te + a.s - 1) / a.s + 1 : 1;
  return a;
}

// Chunking of a range of `tiles` tiles: n = ceil(tiles / tile_batch) UNet calls of bc = ceil(tiles / n) tiles each (the
// last one padded with repeats of the range's last tile), so every call has the same shape
struct TileChunks {
  int64_t n;
  int bc;
};
TileChunks tile_chunks(int64_t tiles, int tile_batch) {
  const int64_t n = (tiles + tile_batch - 1) / tile_batch;
  return {n, n ? int((tiles + n - 1) / n) : 0};
}

// The T-step tiled loop over the own tiles [g0, g1) of B canvases.  d_tiled holds [SampleArgs | x (B,C,H,W) | ...]; the
// workspace is reserved for one chunk (bc tiles of te_y x te_x); eps_store is indexed by global tile.  Per step: the
// own tiles' eps into the store, chunk by chunk, then exchange(user, t, st) when given, then the blend of the pixels the
// own tiles cover.  fdsr_sample_tiled: [0, n_tiles), no exchange, no owner.  Plain stream launches: a chunk's UNet (~5 ms
// at bc = 16, 256^2) keeps the device well behind the host's ~0.3 ms of launch calls.
template <typename T>
int tiled_enqueue(fdsr_ctx* c, const float* cond, float* sr_out, bool has_trace, int B, const TileAxis& ay,
                  const TileAxis& ax, int64_t g0, int64_t g1, const TileChunks& ch, float* eps_store,
                  fdsr_tile_exchange_fn exchange, void* user, const TileOwner* owner, cudaStream_t st) {
  const SampleArgs* args = reinterpret_cast<const SampleArgs*>(c->d_tiled.ptr);
  const uint32_t HW = uint32_t(ay.L) * uint32_t(ax.L);
  const int C = c->bands();
  float* x = reinterpret_cast<float*>(c->d_tiled + 256);
  const int64_t tile_floats = int64_t(C) * ay.te * ax.te;
  const unsigned pack_blocks = unsigned((int64_t(ch.bc) * ay.te * ax.te + 255) / 256);
  T* xin = ch.bc ? reinterpret_cast<T*>(c->d_ws + c->tensors[c->t_xin].off) : nullptr;
  const float* eps_chunk = ch.bc ? reinterpret_cast<const float*>(c->d_ws + c->off_eps) : nullptr;
  // the band of canvases / pixel indices that holds every pixel the own tiles cover: the rows of the range's windows
  // when it lies in one canvas, else its canvases whole (an empty range: one block that updates nothing)
  const int64_t per_canvas = int64_t(ay.n) * ax.n;
  int b0 = 0, nb = B;
  uint32_t p0 = 0, p1 = HW;
  if (g0 == g1) {
    nb = 1, p1 = 0;
  } else if (g0 / per_canvas == (g1 - 1) / per_canvas) {
    b0 = int(g0 / per_canvas), nb = 1;
    p0 = uint32_t(tile_start(ay, int(g0 % per_canvas / ax.n))) * uint32_t(ax.L);
    p1 = uint32_t(tile_start(ay, int((g1 - 1) % per_canvas / ax.n)) + ay.te) * uint32_t(ax.L);
  } else if (g0 != 0 || g1 != int64_t(B) * per_canvas) {
    b0 = int(g0 / per_canvas), nb = int((g1 - 1) / per_canvas) - b0 + 1;
  }
  const dim3 pgrid(std::max(1u, unsigned((uint64_t(p1 - p0) + 255) / 256)), unsigned(nb));
  return sample_chain(
      c, args, x, cond, sr_out, B, HW, has_trace, st,
      [&](int t, int k) {
        for (int64_t i = 0; i < ch.n; ++i) {
          const int64_t tile0 = g0 + i * ch.bc, valid = std::min<int64_t>(ch.bc, g1 - tile0);
          int rc = launch(c, tile_pack_kernel<T>, pack_blocks, 256, 0, st, cond, x, xin, ay, ax, tile0, g1 - 1, ch.bc, C);
          if (!rc) rc = unet_internal<T>(c, t, st, false, true);
          if (rc) return rc;
          // padding slots repeat the last own tile and stay in the workspace: the store holds other ranks' slots
          CUDA_TRY(c, cudaMemcpyAsync(eps_store + tile0 * tile_floats, eps_chunk, size_t(valid) * tile_floats * 4,
                                      cudaMemcpyDeviceToDevice, st));
        }
        if (exchange) {
          const int e = exchange(user, t, st);
          if (e) return fail(c, FDSR_E_INVALID, "the tile exchange callback returned %d at step t = %d", e, t);
        }
        return launch(c, tile_blend_posterior_kernel, pgrid, 256, 0, st, x, eps_store, ay, ax, C, c->post[t], args,
                      int64_t(k + 1), uint32_t(t), t > 0 ? 1 : 0, B, b0, p0, p1, g0, g1);
      },
      owner);
}

// The partition and need rule of fdsr_tiled_plan (include/fdsr.h).  Rank r owns [own_lo(r), own_lo(r + 1)).
int64_t own_lo(int64_t n, int world, int r) {
  return int64_t((unsigned __int128)n * unsigned(r) / unsigned(world));
}

// [lo, hi]: the tiles of one axis whose windows intersect the positions [s, e) (their starts ascend, so they are
// contiguous); lo > hi when there are none
void axis_hits(const TileAxis& a, int s, int e, int& lo, int& hi) {
  lo = a.n, hi = -1;
  for (int j = 0; j < a.n; ++j)
    if (tile_start(a, j) < e && tile_start(a, j) + a.te > s) lo = std::min(lo, j), hi = j;
}

// The tiles of [s0, s1) whose windows intersect U = the union of the windows of [r0, r1), as the range [lo, hi) from
// the first to the last of them (lo == hi == 0: none).  The own tiles of one tile row of U have one contiguous column
// span; the windows meeting it form a rectangle of the tile grid, one g-interval per tile row.
void tiles_needed(const TileAxis& ay, const TileAxis& ax, int64_t r0, int64_t r1, int64_t s0, int64_t s1, int64_t* lo,
                  int64_t* hi) {
  int64_t first = INT64_MAX, last = -1;
  for (int64_t g = r0; g < r1 && s0 < s1;) {
    const int64_t row = g / ax.n, row_end = std::min(r1, (row + 1) * ax.n);  // g .. row_end - 1: one tile row
    const int ty = int(row % ay.n);
    int ya, yb, xa, xb;
    axis_hits(ay, tile_start(ay, ty), tile_start(ay, ty) + ay.te, ya, yb);
    axis_hits(ax, tile_start(ax, int(g - row * ax.n)), tile_start(ax, int(row_end - 1 - row * ax.n)) + ax.te, xa, xb);
    for (int y = ya; y <= yb; ++y) {
      const int64_t base = (row - ty + y) * ax.n;
      const int64_t a = std::max(base + xa, s0), z = std::min(base + xb + 1, s1);
      if (a < z) first = std::min(first, a), last = std::max(last, z);
    }
    g = row_end;
  }
  *lo = last < 0 ? 0 : first;
  *hi = last < 0 ? 0 : last;
}

// The entries of peer q in rank's plan: o = {send lo, send hi, recv lo, recv hi}, all 0 for q == rank
void peer_plan(const TileAxis& ay, const TileAxis& ax, int64_t n, int world, int rank, int q, int64_t* o) {
  o[0] = o[1] = o[2] = o[3] = 0;
  if (q == rank) return;
  const int64_t lo = own_lo(n, world, rank), hi = own_lo(n, world, rank + 1);
  const int64_t qlo = own_lo(n, world, q), qhi = own_lo(n, world, q + 1);
  tiles_needed(ay, ax, qlo, qhi, lo, hi, o, o + 1);      // q needs of ours
  tiles_needed(ay, ax, lo, hi, qlo, qhi, o + 2, o + 3);  // we need of q's
}

// out[0..5 + 4 world): n_tiles, te_y, te_x, own lo, own hi, then per peer q: send lo, send hi, recv lo, recv hi
void tiled_plan(const TileAxis& ay, const TileAxis& ax, int64_t n, int world, int rank, int64_t* out) {
  out[0] = n, out[1] = ay.te, out[2] = ax.te, out[3] = own_lo(n, world, rank), out[4] = own_lo(n, world, rank + 1);
  for (int q = 0; q < world; ++q) peer_plan(ay, ax, n, world, rank, q, out + 5 + 4 * int64_t(q));
}

// Pillow precompute_coeffs + normalize_coeffs_8bpc for the bicubic filter, full-image box
int ensure_bic(fdsr_ctx* c, int in, int out) {
  for (const auto& b : c->bic)
    if (b.in == in && b.out == out) return FDSR_OK;
  const double scale = double(in) / out;
  const double fscale = scale < 1.0 ? 1.0 : scale;
  const double support = 2.0 * fscale;
  const int ksize = int(ceil(support)) * 2 + 1;
  std::vector<int> vmin(out), vcnt(out), taps(size_t(out) * ksize, 0);
  std::vector<double> k(ksize);
  auto filt = [](double x) {
    const double a = -0.5;
    if (x < 0.0) x = -x;
    if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
    if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
    return 0.0;
  };
  for (int xx = 0; xx < out; ++xx) {
    const double center = (xx + 0.5) * scale;
    const double ss = 1.0 / fscale;
    int xmin = int(center - support + 0.5);
    if (xmin < 0) xmin = 0;
    int xmax = int(center + support + 0.5);
    if (xmax > in) xmax = in;
    xmax -= xmin;
    double ww = 0.0;
    for (int x = 0; x < xmax; ++x) {
      k[x] = filt((x + xmin - center + 0.5) * ss);
      ww += k[x];
    }
    for (int x = 0; x < xmax; ++x) {
      if (ww != 0.0) k[x] /= ww;
      taps[size_t(xx) * ksize + x] =
          k[x] < 0 ? int(-0.5 + k[x] * (1 << kBicPrec)) : int(0.5 + k[x] * (1 << kBicPrec));
    }
    vmin[xx] = xmin;
    vcnt[xx] = xmax;
  }
  fdsr_ctx::BicTab b{in, out, ksize};
  int rc = upload(c, b.d_min, vmin);
  if (!rc) rc = upload(c, b.d_cnt, vcnt);
  if (!rc) rc = upload(c, b.d_taps, taps);
  if (!rc) c->bic.push_back(std::move(b));
  return rc;
}
const fdsr_ctx::BicTab* find_bic(const fdsr_ctx* c, int in, int out) {
  for (const auto& b : c->bic)
    if (b.in == in && b.out == out) return &b;
  return nullptr;
}

// The checks fdsr_sample_tiled, fdsr_sample_tiled_part and fdsr_tiled_plan share (c == nullptr: the global error)
int tiled_check(fdsr_ctx* c, int32_t B, int32_t H, int32_t W, int32_t tile_h, int32_t tile_w, int32_t overlap) {
  if (B < 1 || B > 65535) return fail(c, FDSR_E_INVALID, "B must be 1..65535 (got %d)", B);
  if (H < 8 || W < 8) return fail(c, FDSR_E_INVALID, "canvas H and W must be >= 8 (got %dx%d)", H, W);
  if (uint64_t(H) * uint64_t(W) >= (uint64_t(1) << 32))
    return fail(c, FDSR_E_INVALID, "canvas H*W must be below 2^32 (got %dx%d)", H, W);
  if (tile_h < 8 || tile_w < 8 || tile_h % 8 || tile_w % 8)
    return fail(c, FDSR_E_INVALID, "tile sizes must be multiples of 8 and >= 8 (got %dx%d)", tile_h, tile_w);
  if (overlap < 0) return fail(c, FDSR_E_INVALID, "overlap must be >= 0 (got %d)", overlap);
  return FDSR_OK;
}

int tiled_entry_check(fdsr_ctx* c, const float* cond, const float* sr_out, int32_t B, int32_t H, int32_t W,
                      int32_t tile_h, int32_t tile_w, int32_t overlap, int32_t tile_batch) {
  if (!cond || !sr_out) return fail(c, FDSR_E_INVALID, "null argument");
  if (c->cfg.model != FDSR_MODEL_FASTDIFFSR)
    return fail(c, FDSR_E_INVALID, "tiled sampling is implemented for the FastDiffSR model only, not the SR3 baseline");
  int rc = tiled_check(c, B, H, W, tile_h, tile_w, overlap);
  if (rc) return rc;
  if (tile_batch < 1) return fail(c, FDSR_E_INVALID, "tile_batch must be >= 1 (got %d)", tile_batch);
  return check_ready(c);
}

// Reserves the workspace for one chunk, grows d_tiled to [SampleArgs | canvas x | store_bytes] and writes SampleArgs
int tiled_prepare(fdsr_ctx* c, const TileChunks& ch, const TileAxis& ay, const TileAxis& ax, int B, size_t store_bytes,
                  const float* noise, uint64_t seed, float* trace, cudaStream_t st) {
  if (ch.bc) {
    int rc = fdsr_reserve(c, ch.bc, ay.te, ax.te);
    if (rc) return rc;
  }
  CUDA_TRY(c, c->d_tiled.grow(256 + align_up(size_t(B) * c->bands() * ay.L * ax.L * 4, 256) + store_bytes));
  return launch(c, set_args_kernel, 1, 1, 0, st, reinterpret_cast<SampleArgs*>(c->d_tiled.ptr),
                SampleArgs{seed, c->image0, noise, trace});
}
}  // namespace

// =============================================================================== C ABI
extern "C" {

const char* fdsr_global_error(void) { return g_global_error.c_str(); }
const char* fdsr_last_error(const fdsr_ctx* ctx) { return ctx ? ctx->err.c_str() : g_global_error.c_str(); }

int fdsr_create(const fdsr_config* cfg, fdsr_ctx** out) {
  if (!cfg || !out) return fail(nullptr, FDSR_E_INVALID, "null argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(nullptr, FDSR_E_CUDA, "no CUDA device: libfdsr has no CPU fallback");
  fdsr_ctx* c = new fdsr_ctx();
  c->cfg = *cfg;
  cudaGetDevice(&c->device);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, c->device) != cudaSuccess || prop.major != 10) {
    delete c;
    return fail(nullptr, FDSR_E_CUDA, "libfdsr needs an sm_100 (B200) device");
  }
  c->num_sms = prop.multiProcessorCount;
  c->pair = env_hook("FDSR_PAIR", c->pair);
  c->half_tiles = env_hook("FDSR_HALF_TILES", c->half_tiles);
  c->split_n = env_hook("FDSR_SPLIT_N", c->split_n);
  c->epi2 = env_hook("FDSR_EPI2", c->epi2);
  c->tail_help = env_hook("FDSR_TAIL_HELP", c->tail_help);
  c->resid_mma = env_hook("FDSR_RESID_MMA", c->resid_mma);
  c->up_phases = env_hook("FDSR_UP_PHASES", c->up_phases);
  c->fused_tail = env_hook("FDSR_FUSED_TAIL", c->fused_tail);
  c->attn_ref = env_hook("FDSR_ATTN_REF", c->attn_ref);
  if (cfg->dtype < FDSR_DTYPE_FP16 || cfg->dtype > FDSR_DTYPE_FP32) {
    delete c;
    return fail(nullptr, FDSR_E_INVALID, "dtype must be FDSR_DTYPE_FP16, FDSR_DTYPE_BF16 or FDSR_DTYPE_FP32");
  }
  const int rc = build_plan(c);
  if (rc) {
    g_global_error = c->err;
    delete c;
    return rc;
  }
  // the 16-bit kernels' dynamic shared memory limits (the fp32 parity mode uses static shared memory only)
  const cudaError_t ae = cfg->dtype == FDSR_DTYPE_FP32 ? cudaSuccess : with_dtype16(c, [&](auto e) {
    using T = typename decltype(e)::type;
    cudaError_t r = set_conv_attrs<T>();
    for (const HAttn& a : c->attns)  // SelfAttention cores of the SR3 baseline
      if (r == cudaSuccess && a.kind == 1)
        r = cudaFuncSetAttribute(attn_core<T>(a.C).first, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 attn_core<T>(a.C).second);
    return r;
  });
  if (ae != cudaSuccess) {
    delete c;
    return fail(nullptr, FDSR_E_CUDA, "cudaFuncSetAttribute(max dynamic smem) failed: %s", cudaGetErrorString(ae));
  }
  *out = c;
  return FDSR_OK;
}

int fdsr_destroy(fdsr_ctx* c) {
  if (!c) return FDSR_OK;
  c->drop_graphs();
  for (auto& sl : c->slot) {
    if (sl.h_pin) cudaFreeHost(sl.h_pin);
    if (sl.computed) cudaEventDestroy(sl.computed);
    if (sl.copied) cudaEventDestroy(sl.copied);
  }
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  delete c;  // and with it every device buffer
  return FDSR_OK;
}

static int finish_load_weights(fdsr_ctx* c);

int fdsr_load_weights(fdsr_ctx* c, const char* const* names, const float* const* ptrs, const int64_t* numels,
                      int32_t n) {
  if (!c || !names || !ptrs || !numels) return fail(c, FDSR_E_INVALID, "null argument");
  c->host_w.clear();
  for (int i = 0; i < n; ++i) {
    if (!names[i] || !ptrs[i] || numels[i] < 0) return fail(c, FDSR_E_INVALID, "null / negative entry %d", i);
    c->host_w[names[i]] = std::vector<float>(ptrs[i], ptrs[i] + numels[i]);
  }
  return finish_load_weights(c);
}

int fdsr_load_weights_dev(fdsr_ctx* c, const char* const* names, const float* const* dev_ptrs, const int64_t* numels,
                          int32_t n, void* stream) {
  if (!c || !names || !dev_ptrs || !numels) return fail(c, FDSR_E_INVALID, "null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  c->host_w.clear();
  // the pointers are borrowed for the duration of the call: one device -> host copy per tensor into the repacking
  // buffers (the repack itself — tap blobs, FiLM tables — is host code), no round trip through the caller's host memory
  for (int i = 0; i < n; ++i) {
    if (!names[i] || !dev_ptrs[i] || numels[i] < 0) return fail(c, FDSR_E_INVALID, "null / negative entry %d", i);
    std::vector<float>& v = c->host_w[names[i]];
    v.resize(size_t(numels[i]));
    if (numels[i]) CUDA_TRY(c, cudaMemcpyAsync(v.data(), dev_ptrs[i], size_t(numels[i]) * 4, cudaMemcpyDeviceToHost, st));
  }
  CUDA_TRY(c, cudaStreamSynchronize(st));
  return finish_load_weights(c);
}

static int finish_load_weights(fdsr_ctx* c) {
  int rc = validate_weights(c);
  if (rc) {
    c->host_w.clear();
    c->weights_loaded = false;
    return rc;
  }
  rc = with_dtype(c, [&](auto e) {
    using T = typename decltype(e)::type;
    if constexpr (sizeof(T) == 4) return pack_weights_f32(c);
    else return pack_weights<T>(c);
  });
  if (rc) return rc;
  rc = upload_params(c);
  if (rc) return rc;
  c->weights_loaded = true;
  c->layers_dirty = true;
  c->drop_graphs();
  if (c->T) return build_bias_tables(c);
  return FDSR_OK;
}

int fdsr_set_schedule(fdsr_ctx* c, const double* betas, int32_t T) {
  if (!c || !betas || T < 1) return fail(c, FDSR_E_INVALID, "bad schedule");
  if (!c->weights_loaded) return fail(c, FDSR_E_STATE, "load weights before the schedule (FiLM tables need them)");
  std::vector<double> b(betas, betas + T), al(T), ac(T), acp(T), pv(T);
  auto& tb = c->tables;
  tb.clear();
  double cp = 1.0;
  for (int i = 0; i < T; ++i) {
    al[i] = 1.0 - b[i];
    acp[i] = cp;
    cp *= al[i];
    ac[i] = cp;
  }
  std::vector<double> s_ac(T), s_1m(T), l_1m(T), s_r(T), s_rm1(T), plv(T), c1(T), c2(T), nlv(T + 1);
  nlv[0] = 1.0;
  for (int i = 0; i < T; ++i) {
    s_ac[i] = sqrt(ac[i]);
    s_1m[i] = sqrt(1.0 - ac[i]);
    l_1m[i] = log(1.0 - ac[i]);
    s_r[i] = sqrt(1.0 / ac[i]);
    s_rm1[i] = sqrt(1.0 / ac[i] - 1);
    pv[i] = b[i] * (1.0 - acp[i]) / (1.0 - ac[i]);
    plv[i] = log(pv[i] > 1e-20 ? pv[i] : 1e-20);
    c1[i] = b[i] * sqrt(acp[i]) / (1.0 - ac[i]);
    c2[i] = (1.0 - acp[i]) * sqrt(al[i]) / (1.0 - ac[i]);
    nlv[i + 1] = sqrt(ac[i]);
  }
  tb["betas"] = b;
  tb["alphas_cumprod"] = ac;
  tb["alphas_cumprod_prev"] = acp;
  tb["sqrt_alphas_cumprod"] = s_ac;
  tb["sqrt_one_minus_alphas_cumprod"] = s_1m;
  tb["log_one_minus_alphas_cumprod"] = l_1m;
  tb["sqrt_recip_alphas_cumprod"] = s_r;
  tb["sqrt_recipm1_alphas_cumprod"] = s_rm1;
  tb["posterior_variance"] = pv;
  tb["posterior_log_variance_clipped"] = plv;
  tb["posterior_mean_coef1"] = c1;
  tb["posterior_mean_coef2"] = c2;
  tb["sqrt_alphas_cumprod_prev"] = nlv;
  c->T = T;
  c->post.resize(T);
  for (int i = 0; i < T; ++i)
    c->post[i] = PostCoef{float(s_r[i]), float(s_rm1[i]), float(c1[i]), float(c2[i]), expf(0.5f * float(plv[i]))};
  {  // per-step arguments of the fused final-conv epilogue: step t is the (T-1-t)-th of the loop, its z block T-t
    std::vector<PostStep> ps(T);
    for (int t = 0; t < T; ++t) ps[t] = PostStep{c->post[t], T - t, t > 0 ? 1 : 0, {0}};
    c->layers_dirty = true;
    const int rc = upload(c, c->d_post, ps);
    if (rc) return rc;
  }
  c->drop_graphs();
  return build_bias_tables(c);
}

int fdsr_get_table(fdsr_ctx* c, const char* name, double* out, int32_t cap) {
  if (!c || !name || !out) return fail(c, FDSR_E_INVALID, "null argument");
  auto it = c->tables.find(name);
  if (it == c->tables.end()) return fail(c, FDSR_E_NOTFOUND, "no table %s", name);
  if (cap < int(it->second.size())) return fail(c, FDSR_E_INVALID, "capacity too small");
  memcpy(out, it->second.data(), it->second.size() * 8);
  return int(it->second.size());
}

int fdsr_reserve(fdsr_ctx* c, int32_t B, int32_t H, int32_t W) {
  if (!c) return FDSR_E_INVALID;
  const int down = 1 << (c->cfg.n_levels - 1);
  if (B < 1 || H < down || W < down || H % down || W % down)
    return fail(c, FDSR_E_INVALID, "B>=1 and H, W multiples of %d required (got %dx%dx%d)", down, B, H, W);
  if (c->B == B && c->H == H && c->W == W && c->d_ws) return FDSR_OK;
  // per-call sampler arguments and the overflow flag sit at the start so that they never move
  size_t off = 256;
  for (HTensor& t : c->tensors) {
    t.off = off;
    off = align_up(off + size_t(B) * (H >> t.level) * (W >> t.level) * t.C * c->esize(), 256);
  }
  c->stats_off = off;
  for (HTensor& t : c->tensors)
    if (t.stats) {
      t.stats_off = off;
      off += size_t(B) * t.C * 8;
    }
  // CLAM pools live in the per-forward zeroed region too
  int cmax = 0, lmin = 99;
  for (const HAttn& a : c->attns) {
    if (a.kind != 0) continue;
    cmax = a.C > cmax ? a.C : cmax;
    lmin = c->tensors[a.in].level < lmin ? c->tensors[a.in].level : lmin;
  }
  c->off_psum = off;
  off += size_t(B) * cmax * 8;
  c->off_pmax = off;
  off += size_t(B) * cmax * 4;
  off = align_up(off, 256);
  c->stats_bytes = off - c->stats_off;
  c->off_gate = off;
  off = align_up(off + size_t(B) * cmax * 4, 256);
  c->off_sp = off;
  off = align_up(off + (lmin < 99 ? size_t(B) * (H >> lmin) * (W >> lmin) * 8 : 0), 256);
  const size_t img = align_up(size_t(B) * c->bands() * H * W * 4, 256);
  c->off_cond = off;
  off += img;
  c->off_x = off;
  off += img;
  c->off_eps = off;
  off += img;
  c->off_sr = off;
  off += img;
  c->off_seed = 0;
  c->off_gntab = off;
  off += c->cfg.dtype == FDSR_DTYPE_FP32 ? size_t(B) * kMaxGnC * 8 : 0;
  // grow-only: the captured graphs of other shapes hold pointers into the workspace and stay valid as long as it is
  // not reallocated (alternating shapes / a ragged last batch re-use their graphs)
  if (off > c->d_ws.cap) {
    c->drop_graphs();
    CUDA_TRY(c, c->d_ws.grow(off));
    CUDA_TRY(c, cudaMemset(c->d_ws, 0, 256));
  }
  c->ws_bytes = off;
  c->B = B;
  c->H = H;
  c->W = W;
  c->layers_dirty = true;
  return FDSR_OK;
}

size_t fdsr_workspace_bytes(const fdsr_ctx* c) { return c ? c->ws_bytes : 0; }

int fdsr_unet_forward(fdsr_ctx* c, const float* cond, const float* xt, int32_t t, float* eps_out, int32_t B,
                      int32_t H, int32_t W, void* stream) {
  if (!c || !cond || !xt || !eps_out) return fail(c, FDSR_E_INVALID, "null argument");
  int rc = check_ready(c);
  if (rc) return rc;
  if (t < 0 || t >= c->T) return fail(c, FDSR_E_INVALID, "t out of range");
  rc = fdsr_reserve(c, B, H, W);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t bytes = size_t(B) * c->bands() * H * W * 4;
  CUDA_TRY(c, cudaMemcpyAsync(c->d_ws + c->off_cond, cond, bytes, cudaMemcpyDeviceToDevice, st));
  CUDA_TRY(c, cudaMemcpyAsync(c->d_ws + c->off_x, xt, bytes, cudaMemcpyDeviceToDevice, st));
  rc = unet_dispatch(c, t, st);
  if (rc) return rc;
  CUDA_TRY(c, cudaMemcpyAsync(eps_out, c->d_ws + c->off_eps, bytes, cudaMemcpyDeviceToDevice, st));
  return FDSR_OK;
}

int fdsr_posterior_step(fdsr_ctx* c, const float* xt, const float* eps, const float* z, int32_t t, float* out,
                        int64_t numel, void* stream) {
  if (!c || !xt || !eps || !out) return fail(c, FDSR_E_INVALID, "null argument");
  if (c->T == 0) return fail(c, FDSR_E_STATE, "fdsr_set_schedule has not been called");
  if (t < 0 || t >= c->T) return fail(c, FDSR_E_INVALID, "t out of range");
  if (t > 0 && !z) return fail(c, FDSR_E_INVALID, "z is required for t > 0");
  const int C = c->bands();
  if (numel < C || numel % C)
    return fail(c, FDSR_E_INVALID, "numel must be a positive multiple of %d ((B,%d,H,W) tensors)", C, C);
  // elementwise with an explicit z: treated as one (C, numel/C) image (split into equal blocks if it is huge)
  int64_t blocks = 1;
  while (numel % (C * blocks) != 0 || (numel / blocks) / C > 0x7fffffffLL) ++blocks;
  return posterior_launch(c, xt, eps, z, t, out, numel / blocks, int(blocks), nullptr, 0, static_cast<cudaStream_t>(stream));
}

int32_t fdsr_trace_frames(const fdsr_ctx* c) {
  if (!c || c->T == 0) return 0;
  int n = 1;
  for (int t = c->T - 1; t >= 0; --t)
    if (t % trace_every(c->T) == 0) ++n;
  return n;
}

int fdsr_sample(fdsr_ctx* c, const float* cond, const float* noise, uint64_t seed, float* sr_out, float* trace,
                int32_t B, int32_t H, int32_t W, void* stream) {
  if (!c || !cond || !sr_out) return fail(c, FDSR_E_INVALID, "null argument");
  int rc = check_ready(c);
  if (rc) return rc;
  rc = fdsr_reserve(c, B, H, W);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t bytes = size_t(B) * c->bands() * H * W * 4;
  CUDA_TRY(c, cudaMemcpyAsync(c->d_ws + c->off_cond, cond, bytes, cudaMemcpyDeviceToDevice, st));
  // seed, image offset and the noise / trace pointers are read from device memory: one captured graph per shape
  rc = launch(c, set_args_kernel, 1, 1, 0, st, reinterpret_cast<SampleArgs*>(c->d_ws + c->off_seed),
              SampleArgs{seed, c->image0, noise, trace});
  if (rc) return rc;
  // a T = 1000 schedule would be a graph of ~10^5 nodes: long schedules are enqueued directly (the host runs
  // far ahead of the device: ~0.3 ms of launch calls per ~5 ms UNet step)
  const bool want_graph = c->use_graph && c->T <= 100;
  if (want_graph) {
    rc = ensure_layers(c);
    if (rc) return rc;
    fdsr_ctx::GraphEntry* hit = nullptr;
    for (auto& g : c->graphs)
      if (g.B == B && g.H == H && g.W == W && g.noise == (noise != nullptr) && g.trace == (trace != nullptr)) hit = &g;
    if (!hit) {
      constexpr size_t kMaxGraphs = 8;
      if (c->graphs.size() >= kMaxGraphs) {  // evict the least recently used
        size_t lru = 0;
        for (size_t i = 1; i < c->graphs.size(); ++i)
          if (c->graphs[i].used < c->graphs[lru].used) lru = i;
        cudaGraphExecDestroy(c->graphs[lru].exec);
        c->graphs.erase(c->graphs.begin() + lru);
      }
      cudaStream_t cs;
      CUDA_TRY(c, cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
      const int64_t l0 = c->launches;
      CUDA_TRY(c, cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
      rc = sample_enqueue(c, trace != nullptr, cs);
      cudaGraph_t g = nullptr;
      cudaError_t e = cudaStreamEndCapture(cs, &g);
      cudaStreamDestroy(cs);
      const int64_t per_replay = c->launches - l0;
      c->launches = l0;  // captured, not yet launched
      if (rc) {
        if (g) cudaGraphDestroy(g);
        return rc;
      }
      if (e != cudaSuccess) return fail(c, FDSR_E_CUDA, "graph capture failed: %s", cudaGetErrorString(e));
      cudaGraphExec_t exec = nullptr;
      e = cudaGraphInstantiate(&exec, g, 0);
      cudaGraphDestroy(g);
      if (e != cudaSuccess) return fail(c, FDSR_E_CUDA, "graph instantiate failed: %s", cudaGetErrorString(e));
      c->graphs.push_back({B, H, W, noise != nullptr, trace != nullptr, exec, 0, per_replay});
      hit = &c->graphs.back();
      ++c->graph_captures;
    }
    hit->used = ++c->graph_clock;
    CUDA_TRY(c, cudaGraphLaunch(hit->exec, st));
    c->launches += hit->launches;
  } else {
    rc = sample_enqueue(c, trace != nullptr, st);
    if (rc) return rc;
  }
  CUDA_TRY(c, cudaMemcpyAsync(sr_out, c->d_ws + c->off_sr, bytes, cudaMemcpyDeviceToDevice, st));
  return FDSR_OK;
}

int fdsr_sample_tiled(fdsr_ctx* c, const float* cond, const float* noise, uint64_t seed, float* sr_out, float* trace,
                      int32_t B, int32_t H, int32_t W, int32_t tile_h, int32_t tile_w, int32_t overlap,
                      int32_t tile_batch, void* stream) {
  if (!c) return FDSR_E_INVALID;
  int rc = tiled_entry_check(c, cond, sr_out, B, H, W, tile_h, tile_w, overlap, tile_batch);
  if (rc) return rc;
  const TileAxis ay = make_axis(H, tile_h, overlap), ax = make_axis(W, tile_w, overlap);
  const int64_t n_tiles = int64_t(B) * ay.n * ax.n;
  const TileChunks ch = tile_chunks(n_tiles, tile_batch);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // the context's store has a slot for every chunk slot, padding included
  const size_t store_bytes = size_t(ch.n) * ch.bc * c->bands() * ay.te * ax.te * 4;
  rc = tiled_prepare(c, ch, ay, ax, B, store_bytes, noise, seed, trace, st);
  if (rc) return rc;
  float* eps_store = reinterpret_cast<float*>(c->d_tiled + 256 + align_up(size_t(B) * c->bands() * H * W * 4, 256));
  return with_dtype(c, [&](auto e) {
    return tiled_enqueue<typename decltype(e)::type>(c, cond, sr_out, trace != nullptr, B, ay, ax, 0, n_tiles, ch,
                                                     eps_store, nullptr, nullptr, nullptr, st);
  });
}

int64_t fdsr_tiled_plan(int32_t B, int32_t H, int32_t W, int32_t tile_h, int32_t tile_w, int32_t overlap, int32_t world,
                        int32_t rank, int64_t* out_host, int64_t cap) {
  int rc = tiled_check(nullptr, B, H, W, tile_h, tile_w, overlap);
  if (rc) return rc;
  if (world < 1) return fail(nullptr, FDSR_E_INVALID, "world must be >= 1 (got %d)", world);
  if (rank < 0 || rank >= world) return fail(nullptr, FDSR_E_INVALID, "rank must be 0..world-1 (got %d of %d)", rank, world);
  const int64_t need = 5 + 4 * int64_t(world);
  if (!out_host || cap < need)
    return fail(nullptr, FDSR_E_INVALID, "the plan needs %lld entries (5 + 4 * world), cap is %lld", (long long)need,
                (long long)cap);
  const TileAxis ay = make_axis(H, tile_h, overlap), ax = make_axis(W, tile_w, overlap);
  tiled_plan(ay, ax, int64_t(B) * ay.n * ax.n, world, rank, out_host);
  return need;
}

int fdsr_sample_tiled_part(fdsr_ctx* c, const float* cond, const float* noise, uint64_t seed, float* sr_out,
                           float* trace, int32_t B, int32_t H, int32_t W, int32_t tile_h, int32_t tile_w,
                           int32_t overlap, int32_t tile_batch, int32_t rank, int32_t world, float* eps_store,
                           fdsr_tile_exchange_fn exchange, void* user, void* stream) {
  if (!c) return FDSR_E_INVALID;
  int rc = tiled_entry_check(c, cond, sr_out, B, H, W, tile_h, tile_w, overlap, tile_batch);
  if (rc) return rc;
  if (!eps_store) return fail(c, FDSR_E_INVALID, "null argument (eps_store)");
  if (world < 1) return fail(c, FDSR_E_INVALID, "world must be >= 1 (got %d)", world);
  if (rank < 0 || rank >= world) return fail(c, FDSR_E_INVALID, "rank must be 0..world-1 (got %d of %d)", rank, world);
  const TileAxis ay = make_axis(H, tile_h, overlap), ax = make_axis(W, tile_w, overlap);
  const int64_t n_tiles = int64_t(B) * ay.n * ax.n;
  const TileOwner owner{ay, ax, own_lo(n_tiles, world, rank), own_lo(n_tiles, world, rank + 1)};
  for (int q = 0; q < world && !exchange; ++q) {
    int64_t o[4];
    peer_plan(ay, ax, n_tiles, world, rank, q, o);
    if (o[1] > o[0] || o[3] > o[2])
      return fail(c, FDSR_E_INVALID, "rank %d of %d exchanges tiles with rank %d: the exchange callback is required",
                  rank, world, q);
  }
  const TileChunks ch = tile_chunks(owner.g1 - owner.g0, tile_batch);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  rc = tiled_prepare(c, ch, ay, ax, B, 0, noise, seed, trace, st);
  if (rc) return rc;
  return with_dtype(c, [&](auto e) {
    return tiled_enqueue<typename decltype(e)::type>(c, cond, sr_out, trace != nullptr, B, ay, ax, owner.g0, owner.g1,
                                                     ch, eps_store, exchange, user, &owner, st);
  });
}

int fdsr_bicubic_u8(fdsr_ctx* c, const uint8_t* lr, int32_t B, int32_t h, int32_t w, int32_t H, int32_t W,
                    uint8_t* out_u8, float* cond, void* stream) {
  if (!c || !lr) return fail(c, FDSR_E_INVALID, "null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = ensure_bic(c, w, W);
  if (rc) return rc;
  rc = ensure_bic(c, h, H);
  if (rc) return rc;
  const fdsr_ctx::BicTab *th = find_bic(c, w, W), *tv = find_bic(c, h, H);
  const int C = c->bands();
  const size_t tmp = size_t(B) * h * W * C;
  CUDA_TRY(c, c->d_bic_tmp.grow(tmp));
  const int64_t n1 = int64_t(B) * h * W, n2 = int64_t(B) * H * W;
  rc = launch(c, bicubic_h_kernel, unsigned((n1 + 255) / 256), 256, 0, st, lr, c->d_bic_tmp.ptr, th->d_min.ptr,
              th->d_cnt.ptr, th->d_taps.ptr, th->ksize, B, h, w, W, C);
  if (rc) return rc;
  return launch(c, bicubic_v_kernel, unsigned((n2 + 255) / 256), 256, 0, st, c->d_bic_tmp.ptr, out_u8, cond,
                tv->d_min.ptr, tv->d_cnt.ptr, tv->d_taps.ptr, tv->ksize, B, h, H, W, C);
}

int fdsr_super_resolve_u8_submit(fdsr_ctx* c, int32_t slot, const uint8_t* lr_host, int32_t B, int32_t h, int32_t w,
                                 int32_t H, int32_t W, const float* noise_dev, uint64_t seed, void* stream) {
  if (!c || !lr_host || slot < 0 || slot >= fdsr_ctx::kHostSlots) return fail(c, FDSR_E_INVALID, "bad argument");
  int rc = check_ready(c);
  if (rc) return rc;
  fdsr_ctx::HostSlot& sl = c->slot[slot];
  if (sl.busy) return fail(c, FDSR_E_STATE, "slot %d still holds a result: call fdsr_super_resolve_u8_wait first", slot);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!c->copy_stream) CUDA_TRY(c, cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  if (!sl.computed) {
    CUDA_TRY(c, cudaEventCreateWithFlags(&sl.computed, cudaEventDisableTiming));
    CUDA_TRY(c, cudaEventCreateWithFlags(&sl.copied, cudaEventDisableTiming));
  }
  const size_t in_b = size_t(B) * h * w * c->bands(), out_b = size_t(B) * c->bands() * H * W * 4,
               in_a = align_up(in_b, 256);
  const size_t need_pin = in_a + out_b + 256, need_dev = in_a + 2 * out_b + 256;
  if (need_pin > sl.h_pin_bytes) {
    if (sl.h_pin) cudaFreeHost(sl.h_pin);
    sl.h_pin = nullptr;
    sl.h_pin_bytes = 0;
    CUDA_TRY(c, cudaMallocHost(&sl.h_pin, need_pin));
    sl.h_pin_bytes = need_pin;
  }
  CUDA_TRY(c, sl.d_stage.grow(need_dev));
  sl.in_b = in_b;
  sl.out_b = out_b;
  uint8_t* d_lr = sl.d_stage;
  float* d_cond = reinterpret_cast<float*>(sl.d_stage + in_a);
  float* d_sr = reinterpret_cast<float*>(sl.d_stage + in_a + out_b);
  uint8_t* d_flag = sl.d_stage + in_a + 2 * out_b;
  memcpy(sl.h_pin, lr_host, in_b);
  CUDA_TRY(c, cudaMemcpyAsync(d_lr, sl.h_pin, in_b, cudaMemcpyHostToDevice, st));
  rc = fdsr_bicubic_u8(c, d_lr, B, h, w, H, W, nullptr, d_cond, stream);
  if (rc) return rc;
  rc = fdsr_sample(c, d_cond, noise_dev, seed, d_sr, nullptr, B, H, W, stream);
  if (rc) return rc;
  // the batch's own copy of the status word (fp16 overflow flag), then clear it for the next batch
  CUDA_TRY(c, cudaMemcpyAsync(d_flag, c->d_ws + kOffFlags, 4, cudaMemcpyDeviceToDevice, st));
  CUDA_TRY(c, cudaMemsetAsync(c->d_ws + kOffFlags, 0, 4, st));
  CUDA_TRY(c, cudaEventRecord(sl.computed, st));
  // device -> host on the copy stream: overlaps the next batch's sampling on `stream`
  CUDA_TRY(c, cudaStreamWaitEvent(c->copy_stream, sl.computed, 0));
  CUDA_TRY(c, cudaMemcpyAsync(sl.h_pin + in_a, d_sr, out_b, cudaMemcpyDeviceToHost, c->copy_stream));
  CUDA_TRY(c, cudaMemcpyAsync(sl.h_pin + in_a + out_b, d_flag, 4, cudaMemcpyDeviceToHost, c->copy_stream));
  CUDA_TRY(c, cudaEventRecord(sl.copied, c->copy_stream));
  sl.busy = true;
  return FDSR_OK;
}

int fdsr_super_resolve_u8_wait(fdsr_ctx* c, int32_t slot, float* sr_out_host) {
  if (!c || !sr_out_host || slot < 0 || slot >= fdsr_ctx::kHostSlots) return fail(c, FDSR_E_INVALID, "bad argument");
  fdsr_ctx::HostSlot& sl = c->slot[slot];
  if (!sl.busy) return fail(c, FDSR_E_STATE, "slot %d has no batch in flight", slot);
  CUDA_TRY(c, cudaEventSynchronize(sl.copied));
  sl.busy = false;
  const size_t in_a = align_up(sl.in_b, 256);
  unsigned int flags = 0;
  memcpy(&flags, sl.h_pin + in_a + sl.out_b, 4);
  if (flags & 1u)
    return fail(c, FDSR_E_OVERFLOW, "fp16 overflow: an activation exceeded +-65504 and was stored saturated; the result is "
                                    "not trustworthy -- create the context with FDSR_DTYPE_BF16 for this network");
  memcpy(sr_out_host, sl.h_pin + in_a, sl.out_b);
  return FDSR_OK;
}

int fdsr_super_resolve_u8(fdsr_ctx* c, const uint8_t* lr_host, int32_t B, int32_t h, int32_t w, int32_t H, int32_t W,
                          const float* noise_dev, uint64_t seed, float* sr_out_host, void* stream) {
  if (!c || !lr_host || !sr_out_host) return fail(c, FDSR_E_INVALID, "null argument");
  if (c->slot[0].busy) return fail(c, FDSR_E_STATE, "slot 0 holds a pipelined batch: wait for it first");
  int rc = fdsr_super_resolve_u8_submit(c, 0, lr_host, B, h, w, H, W, noise_dev, seed, stream);
  if (rc) return rc;
  return fdsr_super_resolve_u8_wait(c, 0, sr_out_host);
}

int fdsr_sse_u8(fdsr_ctx* c, const float* a, const float* b, int32_t B, int32_t H, int32_t W, double* sse,
                void* stream) {
  if (!c || !a || !b || !sse) return fail(c, FDSR_E_INVALID, "null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_TRY(c, cudaMemsetAsync(sse, 0, size_t(B) * 8, st));
  const int64_t per = int64_t(c->bands()) * H * W;
  int gx = int((per + 256 * 8 - 1) / (256 * 8));
  return launch(c, sse_u8_kernel, dim3(gx > 0 ? gx : 1, B), 256, 0, st, a, b, sse, per);
}

int fdsr_metrics_u8(fdsr_ctx* c, const float* a, const float* b, int32_t B, int32_t H, int32_t W, double ergas_scale,
                    double* out, void* stream) {
  if (!c || !a || !b || !out || B < 1 || H < 1 || W < 1) return fail(c, FDSR_E_INVALID, "bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_TRY(c, c->d_metric.grow(size_t(B) * 32));
  CUDA_TRY(c, cudaMemsetAsync(c->d_metric, 0, size_t(B) * 32, st));
  const int C = c->bands();
  const dim3 grid((W + kSsimTile - 1) / kSsimTile, (H + kSsimTile - 1) / kSsimTile, B * C);
  const int rc = launch(c, metrics_u8_kernel, grid, 256, 0, st, a, b, c->d_metric.ptr, H, W, C);
  if (rc) return rc;
  return launch(c, metrics_finalize_kernel, (B + 127) / 128, 128, 0, st, c->d_metric.ptr, out, B, H, W, C, ergas_scale);
}

int32_t fdsr_debug_num_tensors(const fdsr_ctx* c) { return c ? int32_t(c->tensors.size()) : 0; }
const char* fdsr_debug_tensor_name(const fdsr_ctx* c, int32_t i) {
  return (c && i >= 0 && i < int(c->tensors.size())) ? c->tensors[i].name.c_str() : nullptr;
}

int fdsr_debug_read_tensor(fdsr_ctx* c, const char* name, float* out, int64_t cap, int32_t* C, int32_t* H, int32_t* W,
                           void* stream) {
  if (!c || !name || !out) return fail(c, FDSR_E_INVALID, "null argument");
  if (!c->d_ws) return fail(c, FDSR_E_STATE, "no forward has run");
  for (const HTensor& t : c->tensors)
    if (t.name == name) {
      const int h = c->H >> t.level, w = c->W >> t.level;
      const int64_t n = int64_t(c->B) * h * w * t.C;
      if (cap < n) return fail(c, FDSR_E_INVALID, "capacity too small (%lld needed)", (long long)n);
      const int rc = with_dtype(c, [&](auto e) {
        using T = typename decltype(e)::type;
        return launch(c, nhwc_to_nchw_kernel<T>, unsigned((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream),
                      reinterpret_cast<const T*>(c->d_ws + t.off), out, c->B, h * w, t.C);
      });
      if (rc) return rc;
      if (C) *C = t.C;
      if (H) *H = h;
      if (W) *W = w;
      return FDSR_OK;
    }
  return fail(c, FDSR_E_NOTFOUND, "no tensor named %s", name);
}

int32_t fdsr_debug_num_ops(const fdsr_ctx* c) { return c ? int32_t(c->ops.size()) : 0; }
const char* fdsr_debug_op_name(const fdsr_ctx* c, int32_t i) {
  if (!c || i < 0 || i >= int(c->ops.size())) return nullptr;
  const HOp& op = c->ops[i];
  if (op.kind == 0) return c->convs[op.idx].name.c_str();
  static thread_local std::string nm;
  nm = c->attns[op.idx].name + (c->attns[op.idx].kind == 0 ? ".clam_slam" : ".attn.core");
  return nm.c_str();
}
static double op_flops(const fdsr_ctx* c, int32_t i, bool executed) {
  if (!c || i < 0 || i >= int(c->ops.size()) || c->ops[i].kind != 0) return 0.0;
  const HConv& k = c->convs[c->ops[i].idx];
  const int lvl = k.out >= 0 ? c->tensors[k.out].level : 0;
  return 2.0 * conv_macs(k, executed) * k.cout * double(c->B) * (c->H >> lvl) * (c->W >> lvl);
}
double fdsr_debug_op_flops(const fdsr_ctx* c, int32_t i) { return op_flops(c, i, false); }
double fdsr_debug_op_flops_executed(const fdsr_ctx* c, int32_t i) { return op_flops(c, i, true); }

int fdsr_debug_op_schedule(fdsr_ctx* c, int32_t i, int32_t* out_host, int32_t cap) {
  if (!c || !out_host) return fail(c, FDSR_E_INVALID, "null argument");
  if (i < 0 || i >= int(c->ops.size()) || c->ops[i].kind != 0) return fail(c, FDSR_E_INVALID, "op %d is not a conv", i);
  if (c->cfg.dtype == FDSR_DTYPE_FP32) return fail(c, FDSR_E_INVALID, "the fp32 parity mode has no tile schedule");
  if (c->layers_dirty || c->h_layers.empty()) return fail(c, FDSR_E_STATE, "run fdsr_unet_forward at the shape first");
  if (cap < kOpScheduleFields) return fail(c, FDSR_E_INVALID, "capacity too small (%d needed)", kOpScheduleFields);
  const ConvLayer& l = c->h_layers[c->ops[i].idx];
  const int grid = conv_grid(c, l);
  // the CTA ranges of conv_gemm_kernel: nclusters contiguous, balanced ranges of tile groups (pair mode: groups of
  // tile pairs, CTA r of a pair computing tile 2k + r); split-N CTAs of one range share its tiles
  const int cs = l.pair ? 2 : 1, ngroups = l.ntiles / cs / l.group, nclusters = grid / cs / l.nsplit;
  const int tq = ngroups / nclusters, tr = ngroups - tq * nclusters, tpi = l.tiles_x * l.tiles_y;
  int max_tiles = 0, spans_image = 0, spans_phase = 0;
  for (int cid = 0; cid < nclusters; ++cid) {
    const int units = tq + (cid < tr ? 1 : 0);
    if (units == 0) continue;
    const int tb = (cid * tq + (cid < tr ? cid : tr)) * l.group, te = tb + units * l.group;
    max_tiles = std::max(max_tiles, te - tb);
    const int b0 = tb * cs / tpi, b1 = ((te - 1) * cs + cs - 1) / tpi;  // first and last virtual image of the range
    spans_image |= b0 / l.phases != b1 / l.phases;
    for (int b = b0; b < b1 && l.phases > 1; ++b) spans_phase |= b / l.phases == (b + 1) / l.phases;
  }
  const int32_t v[kOpScheduleFields] = {l.N,     l.pair,  l.tile_h, l.nsplit, l.group,  grid,        l.ntiles,    max_tiles,
                                        l.epi2,  l.tail2, l.nR,     l.nG,     l.phases, l.a_tma,     spans_image, spans_phase,
                                        l.nchunks};
  std::copy(v, v + kOpScheduleFields, out_host);
  return kOpScheduleFields;
}

int fdsr_debug_profile_unet(fdsr_ctx* c, int32_t t, int32_t reps, float* ms_out_host, int32_t cap, void* stream) {
  if (!c || !ms_out_host) return fail(c, FDSR_E_INVALID, "null argument");
  int rc = check_ready(c);
  if (rc) return rc;
  if (!c->d_ws) return fail(c, FDSR_E_STATE, "run fdsr_unet_forward / fdsr_sample once first");
  const int nops = int(c->ops.size());
  if (cap < nops) return fail(c, FDSR_E_INVALID, "capacity too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  rc = ensure_layers(c);
  if (rc) return rc;
  std::vector<cudaEvent_t> ev(size_t(nops) * 2 * reps);
  for (auto& e : ev) CUDA_TRY(c, cudaEventCreate(&e));
  for (int r = 0; r < reps; ++r) {
    CUDA_TRY(c, cudaMemsetAsync(c->d_ws + c->stats_off, 0, c->stats_bytes, st));
    for (int i = 0; i < nops; ++i) {
      const HOp& op = c->ops[i];
      CUDA_TRY(c, cudaEventRecord(ev[(size_t(r) * nops + i) * 2], st));
      rc = with_dtype(c, [&](auto e) {
        using T = typename decltype(e)::type;
        return op.kind == 0 ? launch_conv<T>(c, op.idx, t, st) : launch_attn<T>(c, op.idx, st);
      });
      if (rc) return rc;
      CUDA_TRY(c, cudaEventRecord(ev[(size_t(r) * nops + i) * 2 + 1], st));
    }
  }
  CUDA_TRY(c, cudaStreamSynchronize(st));
  // the first half of the repetitions only brings the GPU to its sustained (power-capped) clocks: a short
  // burst right after an idle period runs ~10 % faster than the same kernels inside a long sampling loop
  const int r0 = reps >= 4 ? reps / 2 : 0;
  for (int i = 0; i < nops; ++i) {
    double acc = 0.0;
    for (int r = r0; r < reps; ++r) {
      float ms = 0.f;
      CUDA_TRY(c, cudaEventElapsedTime(&ms, ev[(size_t(r) * nops + i) * 2], ev[(size_t(r) * nops + i) * 2 + 1]));
      acc += ms;
    }
    ms_out_host[i] = float(acc / (reps - r0));
  }
  for (auto& e : ev) cudaEventDestroy(e);
  return nops;
}

int fdsr_debug_role_cycles(fdsr_ctx* c, int32_t op, int32_t t, int64_t* out_host, int32_t cap, void* stream) {
  if (!c || !out_host) return fail(c, FDSR_E_INVALID, "null argument");
  int rc = check_ready(c);
  if (rc) return rc;
  if (!c->d_ws) return fail(c, FDSR_E_STATE, "run a forward first");
  if (op < 0 || op >= int(c->ops.size()) || c->ops[op].kind != 0) return fail(c, FDSR_E_INVALID, "op is not a conv");
  if (c->cfg.dtype == FDSR_DTYPE_FP32) return fail(c, FDSR_E_INVALID, "role cycles exist for the tensor-core kernel only");
  const int n = c->num_sms * kProfRoles * 8;
  if (cap < n) return fail(c, FDSR_E_INVALID, "capacity too small");
  rc = ensure_layers(c);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_TRY(c, cudaMemsetAsync(c->d_prof, 0, size_t(n) * 8, st));
  rc = with_dtype16(c, [&](auto e) { return launch_conv<typename decltype(e)::type>(c, c->ops[op].idx, t, st); });
  if (rc) return rc;
  CUDA_TRY(c, cudaMemcpyAsync(out_host, c->d_prof, size_t(n) * 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(c, cudaStreamSynchronize(st));
  return n;
}

// In-situ timeline (FDSR_PROFILE builds): `reps` complete UNet evaluations back to back on `stream`, launched exactly as
// the sampler launches them (programmatic dependent launch, no graph), every conv op writing its CTA stamps into its
// own slice; out_host receives [op][num_sms][kProfRoles][8] of the LAST evaluation (ops that are not convs stay zero).
int fdsr_debug_timeline(fdsr_ctx* c, int32_t t, int32_t reps, int64_t* out_host, int64_t cap, void* stream) {
  if (!c || !out_host) return fail(c, FDSR_E_INVALID, "null argument");
  int rc = check_ready(c);
  if (rc) return rc;
  if (!c->d_ws) return fail(c, FDSR_E_STATE, "run a forward first");
  if (c->cfg.dtype == FDSR_DTYPE_FP32) return fail(c, FDSR_E_INVALID, "timelines exist for the tensor-core kernel only");
  const size_t per_op = size_t(c->num_sms) * kProfRoles * 8, n = per_op * c->ops.size();
  if (size_t(cap) < n) return fail(c, FDSR_E_INVALID, "capacity too small");
  rc = ensure_layers(c);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  long long* buf = nullptr;
  CUDA_TRY(c, cudaMalloc(&buf, n * 8));
  for (size_t i = 0; i < c->ops.size(); ++i)
    if (c->ops[i].kind == 0) c->h_layers[c->ops[i].idx].prof = buf + i * per_op;
  cudaError_t e = cudaSuccess;
  for (int r = 0; r < reps && rc == FDSR_OK && e == cudaSuccess; ++r) {
    if (r + 1 == reps) e = cudaMemsetAsync(buf, 0, n * 8, st);
    if (e == cudaSuccess) rc = unet_dispatch(c, t, st, false);
  }
  if (rc == FDSR_OK && e == cudaSuccess) e = cudaMemcpyAsync(out_host, buf, n * 8, cudaMemcpyDeviceToHost, st);
  const cudaError_t e_sync = cudaStreamSynchronize(st);  // (also on failure: nothing may still write into buf when it is freed)
  if (e == cudaSuccess) e = e_sync;
  for (size_t i = 0; i < c->ops.size(); ++i)
    if (c->ops[i].kind == 0) c->h_layers[c->ops[i].idx].prof = c->d_prof;
  cudaFree(buf);
  if (rc) return rc;
  CUDA_TRY(c, e);
  return int(c->ops.size());
}

int fdsr_check_overflow(fdsr_ctx* c, void* stream) {
  if (!c) return FDSR_E_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!c->d_ws) {
    CUDA_TRY(c, cudaStreamSynchronize(st));
    return FDSR_OK;
  }
  unsigned int flags = 0;
  CUDA_TRY(c, cudaMemcpyAsync(&flags, c->d_ws + kOffFlags, 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(c, cudaStreamSynchronize(st));
  if (flags & 1u) {
    CUDA_TRY(c, cudaMemsetAsync(c->d_ws + kOffFlags, 0, 4, st));
    return fail(c, FDSR_E_OVERFLOW, "fp16 overflow: an activation exceeded +-65504 and was stored saturated; the result is "
                                    "not trustworthy -- create the context with FDSR_DTYPE_BF16 for this network");
  }
  return FDSR_OK;
}

int fdsr_set_image_offset(fdsr_ctx* c, uint64_t first_image) {
  if (!c) return FDSR_E_INVALID;
  c->image0 = first_image;
  return FDSR_OK;
}

int fdsr_debug_noise(fdsr_ctx* c, float* out, int32_t B, int32_t H, int32_t W, uint64_t seed, uint64_t first_image,
                     int32_t stream_id, void* stream) {
  if (!c || !out || B < 1 || B > 65535 || H < 1 || W < 1) return fail(c, FDSR_E_INVALID, "bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SampleArgs* slot = nullptr;  // a private argument slot: the workspace may not exist yet
  CUDA_TRY(c, cudaMallocAsync(reinterpret_cast<void**>(&slot), sizeof(SampleArgs), st));
  const uint32_t hw = uint32_t(H) * uint32_t(W);
  int rc = launch(c, set_args_kernel, 1, 1, 0, st, slot, SampleArgs{seed, first_image, nullptr, nullptr});
  if (!rc)
    rc = launch(c, noise_init_kernel, dim3((hw + 255) / 256, B), 256, 0, st, out, hw, c->bands(), slot, uint32_t(stream_id));
  CUDA_TRY(c, cudaFreeAsync(slot, st));
  return rc;
}

int64_t fdsr_graph_captures(const fdsr_ctx* c) { return c ? c->graph_captures : 0; }

int64_t fdsr_launch_count(const fdsr_ctx* c) { return c ? c->launches : 0; }
double fdsr_unet_flops(const fdsr_ctx* c) { return c ? c->flops_per_px * double(c->B) * c->H * c->W : 0.0; }
int fdsr_set_use_graph(fdsr_ctx* c, int32_t enable) {
  if (!c) return FDSR_E_INVALID;
  c->use_graph = enable != 0;
  return FDSR_OK;
}

}  // extern "C"
