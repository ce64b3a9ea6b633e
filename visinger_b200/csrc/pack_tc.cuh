// Weight pre-pack for the bf16 tensor-core path (implemented in conv_tc.cu).
#pragma once
#include "vsg_common.cuh"

namespace vsg {
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
