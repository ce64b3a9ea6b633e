// Shared host-side plumbing of the C-ABI library: error reporting, the pack object,
// the workspace bump allocator.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda.h>
#include <stdint.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <algorithm>
#include <map>
#include <string>
#include <vector>

#include "../../include/visinger_b200.h"

namespace vsg {

extern thread_local char g_err[1024];
extern thread_local int g_launches;
// launches of conv_tc_kernel per epilogue image (EPI_SIG_*, conv_tc.cuh) since the last reset: the tests read them to see
// which images a call ran
constexpr int kImageSlots = 16;
extern thread_local int g_image_launches[kImageSlots];
inline void reset_launch_counts() {
  g_launches = 0;
  memset(g_image_launches, 0, sizeof(g_image_launches));
}

inline int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define VSG_CUDA_TRY(expr)                                                                         \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess)                                                                         \
      return ::vsg::fail(VSG_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

#define VSG_TRY(expr)            \
  do {                           \
    int _r = (expr);             \
    if (_r != VSG_OK) return _r; \
  } while (0)

#define VSG_LAUNCH_CHECK(what)                                                                    \
  do {                                                                                            \
    ++::vsg::g_launches;                                                                          \
    cudaError_t _e = cudaGetLastError();                                                          \
    if (_e != cudaSuccess)                                                                        \
      return ::vsg::fail(VSG_ECUDA, "launch of %s failed: %s", what, cudaGetErrorString(_e));     \
  } while (0)

// ---- packed weights -----------------------------------------------------------------------------
// fp32 path: [Cin][ktaps][CoutP] + bias[CoutP]
struct ConvW32 {
  float* w = nullptr;
  float* bias = nullptr;
  int Cin = 0, Cout = 0, CoutP = 0, ktaps = 0;
};

// bf16 tensor-core path: [ktaps][CoutT][CinT] bf16 (K-major rows of CinT channels), bias fp32 [CoutT]
struct ConvWTC {
  __nv_bfloat16* w = nullptr;
  float* bias = nullptr;
  int Cin = 0, Cout = 0, CinT = 0, CoutT = 0, ktaps = 0;
  CUtensorMap tmap;     // 2-D map over [ktaps*CoutT rows][CinT]
  bool has_tmap = false;
  bool x3 = false;      // split-bf16 pack: rows are [W_hi (Cin) | W_lo (Cin)], CinT = 2*Cin
  int planes = 1;       // bf16 planes per weight: 1 plain, 2 = x3, 3 = [W_hi | W_mid | W_lo] (the fp32 weight exactly)
  bool wsplit = false;  // planes == 2 pack used with ONE-plane activations: x * W_hi + x * W_lo (weights at ~16 mantissa bits)
};

struct UpsPhase {
  ConvW32 f32;
  ConvWTC tc, x3;
  int in_off0 = 0;
};

struct FlowLayer {
  ConvW32 pre[2], post[2];          // [0] = as stored, [1] = Flip folded in
  std::vector<ConvW32> in_layers;   // gate-interleaved output channels
  std::vector<ConvW32> res_skip;
  float* cond_w = nullptr;          // [2H*n_layers][gin], rows gate-interleaved per layer
  float* cond_b = nullptr;
  // bf16 tensor-core packs
  ConvWTC pre_tc[2], post_tc[2];
  std::vector<ConvWTC> in_tc;       // gate-interleaved
  std::vector<ConvWTC> res_tc;      // res_skip rows [0, H): the residual half (absent for the last layer)
  std::vector<ConvWTC> skip_tc;     // res_skip rows [H, 2H) (all H rows for the last layer)
  // the same packs on three bf16 planes per weight: the flow at the fp32 tolerance on the tensor cores (flow only)
  ConvWTC pre_x6[2], post_x6[2];
  std::vector<ConvWTC> in_x6, res_x6, skip_x6;
  // merged launches (flow only): the WaveNet state h and the skip sum live side by side in one tensor [.., h (H) | out (H)],
  // so res_skip_layers[i] (encoder.py:160-164) runs as the ONE Conv1d(H -> 2H) it is in the reference, and `pre` is
  // zero-extended to 2H output channels so that it also clears the skip sum.  [0] plain bf16, [1] three planes.
  ConvWTC pre2_tc[2][2];            // [flipped][planes == 3]
  std::vector<ConvWTC> rs_tc[2];    // layers 0 .. n_layers - 2
};

// PosteriorEncoder (modules/visinger/encoder.py:76-101): pre (1x1) -> WaveNet -> proj (1x1) -> reparameterised sample.
struct EncPack {
  int in_channels = 0, out_channels = 0, hidden = 0, kernel = 0, dil_rate = 1, n_layers = 0, gin = 0;
  int in_pad = 0;                   // in_channels rounded up to a multiple of 64: row width of the bf16 channels-last input
  ConvW32 pre, proj;
  FlowLayer wn;                     // in_layers / res_skip / cond and their tensor-core packs (pre / post unused)
  std::vector<ConvWTC> pre_tc;      // pre split into input-channel slabs of <= 1024 channels (the kernel's chunk table)
  std::vector<int> pre_c0;          // first input channel of each slab
  ConvWTC proj_tc;
};

// RelativeEncoder (modules/rel_transformer.py:257-320): n_layers x {windowed relative-position self-attention, channel
// LayerNorm, FFN (Conv1d k -> ReLU -> Conv1d 1), LayerNorm}, optional condition through pre_net.
struct RelEncLayer {
  ConvW32 qkv, o, ffn1, ffn2;          // conv_q | conv_k | conv_v stacked into one 1x1 convolution H -> 3H
  ConvWTC qkv_tc, o_tc, ffn1_tc, ffn2_tc;
  float *ek = nullptr, *ev = nullptr;  // emb_rel_k / emb_rel_v [2w+1][dk]
  float *g1 = nullptr, *b1 = nullptr, *g2 = nullptr, *b2 = nullptr;   // LayerNorm gamma / beta
};
struct RelEncPack {
  int hidden = 0, filter = 0, n_heads = 0, n_layers = 0, kernel = 0, window = 0, gin = 0;
  std::vector<RelEncLayer> layers;
  ConvW32 pre_net;                     // Conv1d(gin -> hidden, 1) as a convolution (per-frame condition)
  float *pre_w = nullptr, *pre_b = nullptr;   // the same weights [hidden][gin] for the per-utterance GEMV
  // FramePriorNetwork head: proj = Conv1d(hidden -> 2 hidden, 1) (modules/visinger/encoder.py:65); absent if proj_w is null
  float *proj_w = nullptr, *proj_b = nullptr; // [2H][H], [2H]
  ConvWTC proj_tc;
};

struct ResBlockPack {
  int kernel = 0;
  std::vector<int> dilations;
  std::vector<ConvW32> c1, c2;      // ResBlock2 uses c1 only
  std::vector<ConvWTC> c1_tc, c2_tc;
  std::vector<ConvWTC> c1_x3, c2_x3;   // split-bf16 packs
  std::vector<ConvWTC> c1_rp, c2_rp;   // row-packed block-Toeplitz packs of the dilation-1 convolutions (C <= 32; rp_tc.cuh)
  std::vector<ConvWTC> c1_rp_x3, c2_rp_x3;   // the same as split-bf16 packs [W_hi | W_lo] (bf16x3 mode)
  std::vector<float*> c2_bsum;         // running bias of the residual stream: b2_0 + ... + b2_q, fp32 [C] each (rp_tc.cuh)
};

struct UpStage {
  int rate = 0, kernel = 0, Cin = 0, Cout = 0, pad = 0;
  std::vector<UpsPhase> phases;
  // all `rate` polyphase sub-convolutions as ONE Conv1d(Cin -> rate*Cout): phase r owns output channels
  // [r*Cout, (r+1)*Cout), taps zero-padded to a common window; its [B, L, rate*Cout] output IS [B, L*rate, Cout]
  ConvWTC merged_tc, merged_x3;
  int merged_in_off0 = 0;
  std::vector<ResBlockPack> blocks;
};

// The linear spectrogram of vsg_model_convert (spec.cuh): Conv1d(hop -> 2 * bins, taps) over rows of hop samples with
// the window-folded DFT basis as weights -- output channels (2k, 2k + 1) = (w[n] cos(2 pi k n / n_fft),
// -w[n] sin(2 pi k n / n_fft)) at n = lead + tap * hop + j, lead = (n_fft - win) / 2, zero beyond the window.
struct SpecPack {
  int n_fft = 0, win = 0, hop = 0, bins = 0, taps = 0;
  int off = 0;                         // first sample of frame 0's window: (n_fft - win) / 2 - (n_fft - hop) / 2
  int hopP = 0;                        // hop rounded up to 64: channels of a bf16 row
  ConvW32 f32;                         // Cin = hop, Cout = 2 * bins
  ConvWTC tc;                          // Cin = hopP, Cout = 2 * in_pad of the posterior (pad pairs zero)
};

// The whole model (vsg_model_pack_create): the four sub-packs of the existing pack types plus the token-rate weights that
// no stack owns.  Device arrays live in the owning VsgPack's `allocs`; the sub-packs are destroyed with it.
struct ModelPack {
  VsgModelConfig cfg;
  VsgPack *text = nullptr, *pitch = nullptr, *prior = nullptr, *hot = nullptr;
  const float *ph_emb = nullptr, *pitch_emb = nullptr, *dur_emb = nullptr;   // [n][H]
  const float* lin_wt = nullptr;       // text_encoder.linear.weight transposed: [3H][H]
  const float* lin_b = nullptr;        // [H]
  const float* spk_id_w = nullptr;     // spk_id_proj.weight [num_spk][gin]
  const float *spk_embed_w = nullptr, *spk_embed_b = nullptr;   // spk_embed_proj: [gin][spk_embed_dim], [gin]
  const float *pitch_w = nullptr, *pitch_b = nullptr;           // pitch_predictor.linear: [2][H], [2]
  const float* freq = nullptr;         // embed_positions.freq [H/2], or null: computed on the device
  int gin = 0;
  // voice conversion (vsg_convert_pack_create): the posterior_encoder.* pack and the spectrogram; post is null otherwise
  VsgPack* post = nullptr;
  SpecPack spec;
};
void model_pack_free(ModelPack* m);

}  // namespace vsg

struct VsgPack {
  vsg::ModelPack* model = nullptr;
  VsgConfig cfg;
  int device = 0;
  int hop = 0;
  int sm_count = 148;
  bool has_flow = false, has_dec = false, has_enc = false, has_relenc = false;
  vsg::EncPack enc;
  vsg::RelEncPack relenc;
  std::vector<void*> allocs;
  // flow
  std::vector<vsg::FlowLayer> flow_layers;
  float* flow_cond_w = nullptr;  // cond_layer of every flow stacked: [n_flows * 2H * n_layers][gin] (one GEMV launch)
  float* flow_cond_b = nullptr;
  // decoder
  vsg::ConvW32 conv_pre;
  vsg::ConvWTC conv_pre_tc, conv_pre_x3;
  float* dec_cond_w = nullptr;   // [uic][gin]
  float* dec_cond_b = nullptr;
  std::vector<vsg::UpStage> ups;
  float* conv_post_w = nullptr;  // [C_last][k]
  vsg::ConvWTC conv_post_rp;        // conv_post as a row-packed tensor-core conv: Conv1d(64 -> 16, 3 row taps) over rows of 64 / C_last samples
  vsg::ConvWTC conv_post_rp_x3;  // the same for the bf16x3 stage output (rows of 2 samples x 2 planes x 16 channels, 5 row taps)
  int conv_post_S = 0;           // samples per packed row (0: shape not taken; CUDA-core kernel)
  int conv_post_k = 7;
};

namespace vsg {

struct Workspace {
  char* base;
  size_t cap, off = 0;
  bool overflow = false;
  Workspace(void* p, size_t bytes) : base((char*)p), cap(bytes) {}
  template <typename T>
  T* take(size_t n) {
    size_t bytes = (n * sizeof(T) + 255) & ~(size_t)255;
    if (off + bytes > cap) { overflow = true; off += bytes; return nullptr; }
    T* r = reinterpret_cast<T*>(base + off);
    off += bytes;
    return r;
  }
};

inline size_t align256(size_t n) { return (n + 255) & ~(size_t)255; }

// Makes `dev` current for the scope of a run call and restores the caller's device.
struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

}  // namespace vsg
