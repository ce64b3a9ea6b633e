// fp32 (parity-mode) kernels: CUDA-core FFMA implicit convolution with fused epilogues,
// plus the small non-GEMM glue kernels.  Layout: the reference's own [B, C, T] fp32,
// time contiguous, so this path needs no transposes at the boundary.
//
// One generic kernel covers every convolution on the path:
//   y[b, co, q*out_stride + out_phase] = epi( sum_{ci, j} w[ci][j][co] * f(x[b, ci, q + in_off0 + j*dil]) )
//   * Conv1d (modules/visinger/encoder.py:150-164, decoder.py:72-87): out_stride 1, in_off0 = -padding;
//   * ConvTranspose1d (decoder.py:24-26) as `stride` polyphase sub-convolutions, one launch per phase;
//   * f = leaky_relu on load when the reference applies F.leaky_relu to the conv input
//     (decoder.py:45,55,93,97,126);
//   * epi = the op the reference runs right after the conv: gate (encoder.py:206-213), residual/skip
//     routing (encoder.py:188-194), coupling (flow.py:78,83), residual add / resblock mean (decoder.py:
//     48-54,102);
//   * MAG (template flag): channel pairs (re, im) -> sqrt(re^2 + im^2 + 1e-6) * mask, the linear spectrogram (spec.cuh).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace vsg {

enum : int { EPI_LINEAR = 0, EPI_GATE = 1, EPI_RES_SKIP = 2, EPI_COUPLE = 3 };
enum : int { ACC_SET = 0, ACC_ADD = 1, ACC_ADD_DIV = 2 };

struct ConvF32 {
  // input [B, Cin, Lin]
  const float* x; long long x_bs; int x_cs;
  int Cin, Lin;
  int in_off0, dil, ktaps;
  int pre_lrelu; float slope;
  // weights [Cin][ktaps][CoutP] (CoutP multiple of 64, zero padded), bias [CoutP] or null
  const float* w; int CoutP;
  const float* bias;
  const float* bcond; int bcond_bs;   // per-(batch, out channel) additive term, or null
  int Cout;
  int Lq;
  int out_stride, out_phase, Lout;
  int epi;
  float* y; long long y_bs; int y_cs;
  const float* res; long long res_bs; int res_cs;
  float* y2; long long y2_bs; int y2_cs;
  const float* mask; int mask_bs;     // [B, Lout] or null
  int acc_mode; float acc_div;
  int rs_split;      // EPI_RES_SKIP: channels [0, rs_split) update the state, the rest go to the skip sum
  int y2_first;      // EPI_RES_SKIP: skip sum is written, not accumulated (first layer)
  int y2_mask;       // EPI_RES_SKIP: multiply the skip sum by the mask (last layer)
  int couple_sign;   // EPI_COUPLE: +1 forward (x1 = m + x1*mask), -1 reverse (x1 = (x1 - m)*mask); x1 from res if set
};

constexpr int F32_CI_CHUNK = 8;

__device__ __forceinline__ float lrelu(float v, float slope) { return v > 0.f ? v : v * slope; }
__device__ __forceinline__ float sigmoid_accurate(float v) { return 1.0f / (1.0f + expf(-v)); }

template <int WARPS_CO, int WARPS_Q, bool MAG = false>
__global__ void __launch_bounds__(256) conv_f32_kernel(const ConvF32 p) {
  constexpr int CO_TILE = 8 * WARPS_CO;
  constexpr int Q_TILE = 256 * WARPS_Q;
  static_assert(WARPS_CO * WARPS_Q == 8, "8 warps per CTA");
  extern __shared__ float smem[];
  const int halo = (p.ktaps - 1) * p.dil;
  const int XW = Q_TILE + halo;
  float* xs = smem;                        // [CI_CHUNK][XW]
  float* ws = smem + F32_CI_CHUNK * XW;    // [CI_CHUNK][ktaps][CO_TILE]

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wco = warp % WARPS_CO, wq = warp / WARPS_CO;
  const int b = blockIdx.z, co0 = blockIdx.y * CO_TILE, q0 = blockIdx.x * Q_TILE;

  float acc[8][8];
#pragma unroll
  for (int c = 0; c < 8; ++c)
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[c][i] = 0.f;

  const float* xb = p.x + (long long)b * p.x_bs;
  const int wrow = p.ktaps * CO_TILE;

  for (int ci0 = 0; ci0 < p.Cin; ci0 += F32_CI_CHUNK) {
    // ---- stage the input window (zero padded, optional leaky_relu) ----
    for (int ci = 0; ci < F32_CI_CHUNK; ++ci) {
      const bool cok = (ci0 + ci) < p.Cin;
      const float* xr = xb + (long long)(ci0 + ci) * p.x_cs;
      for (int i = tid; i < XW; i += 256) {
        const int pos = q0 + p.in_off0 + i;
        float v = 0.f;
        if (cok && pos >= 0 && pos < p.Lin) v = __ldg(xr + pos);
        if (p.pre_lrelu) v = lrelu(v, p.slope);
        xs[ci * XW + i] = v;
      }
    }
    // ---- stage the weights of this ci chunk ----
    for (int idx = tid; idx < F32_CI_CHUNK * wrow; idx += 256) {
      const int ci = idx / wrow, rem = idx - ci * wrow;
      const int j = rem / CO_TILE, c = rem - j * CO_TILE;
      float v = 0.f;
      if ((ci0 + ci) < p.Cin && (co0 + c) < p.CoutP)
        v = __ldg(p.w + ((long long)(ci0 + ci) * p.ktaps + j) * p.CoutP + co0 + c);
      ws[idx] = v;
    }
    __syncthreads();
#pragma unroll 1
    for (int ci = 0; ci < F32_CI_CHUNK; ++ci) {
      const float* xrow = xs + ci * XW + wq * 256 + lane;
      const float* wr = ws + ci * wrow + wco * 8;
#pragma unroll 1
      for (int j = 0; j < p.ktaps; ++j) {
        const float4 w0 = *reinterpret_cast<const float4*>(wr + j * CO_TILE);
        const float4 w1 = *reinterpret_cast<const float4*>(wr + j * CO_TILE + 4);
        const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
        float xv[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) xv[i] = xrow[j * p.dil + 32 * i];
#pragma unroll
        for (int c = 0; c < 8; ++c)
#pragma unroll
          for (int i = 0; i < 8; ++i) acc[c][i] = fmaf(wv[c], xv[i], acc[c][i]);
      }
    }
    __syncthreads();
  }

  // ---- fused epilogue ----
  const int cbase = co0 + wco * 8;
  const float* mrow = p.mask ? p.mask + (long long)b * p.mask_bs : nullptr;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int q = q0 + wq * 256 + lane + 32 * i;
    const int n = q * p.out_stride + p.out_phase;
    if (q >= p.Lq || n >= p.Lout) continue;
    const float mk = mrow ? mrow[n] : 1.0f;
    if constexpr (MAG) {   // y[b, c, n] = |(acc[2c], acc[2c + 1])| * mask (no bias)
#pragma unroll
      for (int c = 0; c < 8; c += 2) {
        const int co = cbase + c;
        if (co >= p.Cout) continue;
        const float a = acc[c][i], s = acc[c + 1][i];
        p.y[(long long)b * p.y_bs + (long long)(co >> 1) * p.y_cs + n] = sqrtf(fmaf(a, a, fmaf(s, s, 1e-6f))) * mk;
      }
    } else if (p.epi == EPI_GATE) {
#pragma unroll
      for (int c = 0; c < 8; c += 2) {
        const int co = cbase + c;
        if (co >= p.Cout) continue;
        float a = acc[c][i], s = acc[c + 1][i];
        if (p.bias) { a += p.bias[co]; s += p.bias[co + 1]; }
        if (p.bcond) { a += p.bcond[(long long)b * p.bcond_bs + co]; s += p.bcond[(long long)b * p.bcond_bs + co + 1]; }
        p.y[(long long)b * p.y_bs + (long long)(co >> 1) * p.y_cs + n] = tanhf(a) * sigmoid_accurate(s);
      }
    } else {
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int co = cbase + c;
        if (co >= p.Cout) continue;
        float v = acc[c][i];
        if (p.bias) v += p.bias[co];
        if (p.bcond) v += p.bcond[(long long)b * p.bcond_bs + co];
        if (p.epi == EPI_LINEAR) {
          if (p.res) v += p.res[(long long)b * p.res_bs + (long long)co * p.res_cs + n];
          v *= mk;
          float* yp = p.y + (long long)b * p.y_bs + (long long)co * p.y_cs + n;
          if (p.acc_mode == ACC_ADD) v = *yp + v;
          else if (p.acc_mode == ACC_ADD_DIV) v = (*yp + v) / p.acc_div;
          *yp = v;
        } else if (p.epi == EPI_RES_SKIP) {
          if (co < p.rs_split) {
            float* yp = p.y + (long long)b * p.y_bs + (long long)co * p.y_cs + n;
            *yp = (*yp + v) * mk;
          } else {
            float* yp = p.y2 + (long long)b * p.y2_bs + (long long)(co - p.rs_split) * p.y2_cs + n;
            float o = p.y2_first ? v : (*yp + v);
            if (p.y2_mask) o *= mk;
            *yp = o;
          }
        } else {  // EPI_COUPLE
          // (res != null: the old x1 is read from there -- a flow's first touch of the caller's input -- instead of y)
          const float m = v * mk;
          float* yp = p.y + (long long)b * p.y_bs + (long long)co * p.y_cs + n;
          const float x1 = p.res ? p.res[(long long)b * p.res_bs + (long long)co * p.res_cs + n] : *yp;
          *yp = p.couple_sign > 0 ? (m + x1 * mk) : ((x1 - m) * mk);
        }
      }
    }
  }
}

// ---- speaker-condition projections: out[b, o] = bias[o] + sum_i W[o, i] * g[b, i] -------------
// (WaveNet.cond_layer, encoder.py:171-172, and Generator.cond, decoder.py:42-43: 1x1 convs on a
//  length-1 sequence, i.e. one GEMV per utterance.)  One warp per output element.
__global__ void cond_gemv_kernel(const float* __restrict__ W, const float* __restrict__ bias,
                                 const float* __restrict__ g, float* __restrict__ out, int O, int I, int B) {
  const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (gw >= O * B) return;
  const int b = gw / O, o = gw - b * O;
  const float* wr = W + (long long)o * I;
  const float* gr = g + (long long)b * I;
  float s = 0.f;
  for (int i = lane; i < I; i += 32) s = fmaf(wr[i], gr[i], s);
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
  if (lane == 0) out[(long long)b * O + o] = s + (bias ? bias[o] : 0.f);
}

// ---- prior sampling, models/visinger.py:107 ---------------------------------------------------
__global__ void prior_sample_kernel(const float* __restrict__ mu, const float* __restrict__ logs,
                                    const float* __restrict__ noise, const float* __restrict__ mask,
                                    float* __restrict__ z, int C, int T, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long bt = i / ((long long)C * T);
  const int t = (int)(i % T);
  z[i] = (mu[i] + noise[i] * expf(logs[i])) * mask[bt * T + t];
}

// ---- posterior sampling, modules/visinger/encoder.py:96-97: z = (mu + noise * exp(logs)) * mask with mu / logs the two
// channel halves of stats [B, 2C, T]
__global__ void posterior_sample_kernel(const float* __restrict__ stats, const float* __restrict__ noise,
                                        const float* __restrict__ mask, float* __restrict__ z, int C, int T, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long CT = (long long)C * T;
  const long long b = i / CT, r = i - b * CT;
  const int t = (int)(r % T);
  const float mu = stats[b * 2 * CT + r], logs = stats[b * 2 * CT + CT + r];
  z[i] = (mu + noise[i] * expf(logs)) * mask[b * T + t];
}

// ---- y = x * mask (z_q * mask before the decoder, models/visinger.py:109-111) -----------------
__global__ void mask_mul_kernel(const float* __restrict__ x, const float* __restrict__ mask, float* __restrict__ y,
                                int C, int T, long long total, int mask_ld) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long bt = i / ((long long)C * T);
  const int t = (int)(i % T);
  y[i] = x[i] * mask[bt * mask_ld + t];
}

// ---- channel flip (only needed when n_flows is odd: the folded flips do not cancel) -----------
__global__ void flip_channels_kernel(float* __restrict__ x, int C, int T, long long total_half) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total_half) return;
  const int t = (int)(i % T);
  const long long r = i / T;
  const int c = (int)(r % (C / 2));
  const long long b = r / (C / 2);
  float* lo = x + (b * C + c) * T + t;
  float* hi = x + (b * C + (C - 1 - c)) * T + t;
  const float a = *lo; *lo = *hi; *hi = a;
}

// ---- conv_post (C -> 1, k taps, no bias) fused with the leading leaky_relu and trailing tanh --
// decoder.py:55-57.  One thread per output sample; reads are coalesced along time.  Samples [n0, n1) of each utterance go
// to wav rows wav_ld apart (the whole output: 0, L, L; a streaming window: its central samples).
__global__ void conv_post_f32_kernel(const float* __restrict__ x, const float* __restrict__ w /*[C][k]*/,
                                     float* __restrict__ wav, int C, int L, int k, float slope, int n0, int n1,
                                     long long wav_ld) {
  extern __shared__ float wsm[];
  for (int i = threadIdx.x; i < C * k; i += blockDim.x) wsm[i] = w[i];
  __syncthreads();
  const int n = n0 + blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
  if (n >= n1) return;
  const int pad = (k - 1) / 2;
  const float* xb = x + (long long)b * C * L;
  float s = 0.f;
  for (int c = 0; c < C; ++c) {
    const float* xr = xb + (long long)c * L;
    for (int j = 0; j < k; ++j) {
      const int pos = n + j - pad;
      if (pos >= 0 && pos < L) s = fmaf(wsm[c * k + j], lrelu(xr[pos], slope), s);
    }
  }
  wav[(long long)b * wav_ld + (n - n0)] = tanhf(s);
}

}  // namespace vsg
