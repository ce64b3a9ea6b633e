// Weight pre-pack: the fp32 FFMA pack (here), and the bf16 tensor-core packs (implemented in run_tc.cu).
#pragma once
#include "vsg_common.cuh"

namespace vsg {
// Host vector -> a device copy owned by P (freed with it).
template <typename T>
int upload(VsgPack* P, const std::vector<T>& h, T** d) {
  void* p = nullptr;
  VSG_CUDA_TRY(cudaMalloc(&p, h.size() * sizeof(T) + 256));
  P->allocs.push_back(p);
  VSG_CUDA_TRY(cudaMemcpy(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
  *d = (T*)p;
  return VSG_OK;
}

inline int round_up(int a, int b) { return (a + b - 1) / b * b; }

struct Identity { int operator()(int c) const { return c; } };
// The gate's tanh / sigmoid halves (encoder.py:206-213) as interleaved output channels: c < H -> 2c, c >= H -> 2(c - H) + 1,
// so one thread of the fp32 kernel owns both halves of an output channel.
struct GateInterleave { int H; int operator()(int c) const { return c < H ? 2 * c : 2 * (c - H) + 1; } };

// Conv1d weight W[co][ci][j] -> fp32 pack [ci][j][CoutP] (CoutP = Cout rounded up to 64, zero padded) + bias [CoutP],
// output channel co stored at perm(co).
template <typename Perm>
int pack_conv_f32(VsgPack* P, const std::vector<float>& W, const std::vector<float>& b, int Cout, int Cin, int k, Perm perm,
                  ConvW32* out) {
  out->Cin = Cin; out->Cout = Cout; out->ktaps = k; out->CoutP = round_up(Cout, 64);
  std::vector<float> wp((size_t)Cin * k * out->CoutP, 0.f), bp(out->CoutP, 0.f);
  for (int co = 0; co < Cout; ++co) {
    const int pc = perm(co);
    bp[pc] = b[co];
    for (int ci = 0; ci < Cin; ++ci)
      for (int j = 0; j < k; ++j) wp[((size_t)ci * k + j) * out->CoutP + pc] = W[((size_t)co * Cin + ci) * k + j];
  }
  VSG_TRY(upload(P, wp, &out->w));
  VSG_TRY(upload(P, bp, &out->bias));
  return VSG_OK;
}

// Conv1d-style weight W[co][ci][j] (+ bias[co]) -> bf16 K-major pack and its TMA tensor map.
// planes = 2: split-bf16 pack [W_hi | W_lo] (decoder at the fp32 tolerance); planes = 3: [W_hi | W_mid | W_lo] (flow).
int pack_conv_tc(VsgPack* P, const std::vector<float>& W, const std::vector<float>& b, int Cout, int Cin, int k,
                 ConvWTC* out, int planes = 1);
// ConvTranspose1d(Cin -> Cout, k, stride = rate, padding = (k - rate) / 2), weight W[ci][co][j] (+ bias[co]), as convolutions
// over the input rate: out->phases[r] (outputs q * rate + r: a Conv1d with taps from q + in_off0) and out->merged_* (every
// phase as ONE Conv1d(Cin -> rate * Cout) on a common tap window, zero weights elsewhere), plain and split-bf16.  Fills
// rate / kernel / Cin / Cout / pad; phase_w (optional) receives each phase's Conv1d weight [Cout][Cin][n_r].
int pack_upsampler(VsgPack* P, const std::vector<float>& W, const std::vector<float>& b, int Cin, int Cout, int rate, int k,
                   UpStage* out, std::vector<std::vector<float>>* phase_w = nullptr);
// Dilation-1 Conv1d(C -> C, k), C in {16, 32}, as Conv1d(64 -> 64) over rows of 64 / C time steps with block-Toeplitz
// weights (rp_tc.cuh); leaves out->has_tmap false for shapes the row-packed kernel does not take.
int pack_conv_rowpacked(VsgPack* P, const std::vector<float>& W, int C, int k, ConvWTC* out, int planes = 1);
// rb->c2_bsum[q] = b2[0] + ... + b2[q] on the device (the row-packed kernel keeps the c2 biases out of tensor memory).
int pack_resblock_bias_sums(VsgPack* P, const std::vector<std::vector<float>>& b2, ResBlockPack* rb);
}  // namespace vsg
