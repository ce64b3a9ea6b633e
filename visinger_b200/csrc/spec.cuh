// The linear spectrogram as a convolution (vsg_spectrogram, vsg_model_convert): the kernels around the DFT-basis conv.
//
// Frame f of utterance b covers samples [f*hop - p, f*hop - p + n_fft), p = (n_fft - hop) / 2; its window (win_length
// samples, centred in n_fft as torch.stft pads it) starts at sample f*hop + off, off = (n_fft - win_length) / 2 - p.
// Row r of the framed signal holds samples r*hop + off + j, j < hop, so frame f reads rows f .. f + ktaps - 1 and the
// STFT is Conv1d(hop -> 2 * bins, ktaps) over rows with the window-folded DFT basis as weights (pack: model.cu).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace vsg {
namespace {   // included by run_f32.cu and run_tc.cu: one private copy each

// mask[b, t] = t0 + t < clamp(lengths[b], 0, T_len), t < T: frames [t0, t0 + T) of a T_len-frame batch
__global__ void lengths_mask_kernel(const int32_t* __restrict__ lengths, float* __restrict__ mask, int T, int t0, int T_len,
                                    long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long b = i / T;
  const int t = (int)(i - b * T);
  mask[i] = t0 + t < min(max(lengths[b], 0), T_len) ? 1.f : 0.f;
}

// Sample index s of an utterance of L samples, reflected about its own ends as torch's 'reflect' padding does (no edge
// repeat), folded again for as long as it lies outside [0, L).
__device__ __forceinline__ long long reflect_index(long long s, long long L) {
  if (L <= 1) return 0;
  const long long per = 2 * (L - 1);
  long long m = s % per;
  if (m < 0) m += per;
  return m < L ? m : per - m;
}

// Framed rows r0 .. r0 + R - 1 of every utterance: row r, channel j = wav[b, reflect(r*hop + off + j)] for j < hop and the
// rows that a valid frame f >= r0 reads (r < len + ktaps - 1 and r0 < len, len = clamp(lengths[b], 0, T) frames of
// len * hop samples); 0 elsewhere.  CL: bf16 [B, R, hopP] channels-last (tcgen05 operand), else fp32 [B, hopP, R] (FFMA
// operand).  wav: [B, T * hop], rows wav_ld samples apart; a window (r0 > 0) reads it in place.
template <bool CL>
__global__ void spec_frames_kernel(const float* __restrict__ wav, const int32_t* __restrict__ lengths, void* __restrict__ out,
                                   int T, int R, int hop, int hopP, int off, int ktaps, long long n, int r0, long long wav_ld) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int r, j;
  long long b;
  if (CL) {
    j = (int)(i % hopP);
    const long long br = i / hopP;
    r = (int)(br % R);
    b = br / R;
  } else {
    r = (int)(i % R);
    const long long bj = i / R;
    j = (int)(bj % hopP);
    b = bj / hopP;
  }
  const int len = min(max(lengths[b], 0), T);
  float v = 0.f;
  if (j < hop && r0 + r < len + ktaps - 1 && r0 < len) {
    const long long L = (long long)len * hop;
    v = wav[b * wav_ld + reflect_index((long long)(r0 + r) * hop + off + j, L)];
  }
  if (CL) reinterpret_cast<__nv_bfloat16*>(out)[i] = __float2bfloat16(v);
  else reinterpret_cast<float*>(out)[i] = v;
}

// [B, T, ld] bf16 channels-last -> [B, C, T] fp32 (C <= ld): the tcgen05 spectrogram widened, as the posterior reads it.
__global__ void widen_bf16_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ y, int C, int ld, int T) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, c0 = blockIdx.y * 32, t0 = blockIdx.x * 32;
  const int tx = threadIdx.x, ty = threadIdx.y;   // 32 x 8
  for (int i = ty; i < 32; i += 8) {
    const int t = t0 + i, c = c0 + tx;
    tile[i][tx] = (c < C && t < T) ? __bfloat162float(x[((long long)b * T + t) * ld + c]) : 0.f;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int c = c0 + i, t = t0 + tx;
    if (c < C && t < T) y[((long long)b * C + c) * T + t] = tile[tx][i];
  }
}

}  // namespace
}  // namespace vsg
