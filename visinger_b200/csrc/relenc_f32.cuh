// fp32 (parity-mode) kernels of the relative-position transformer encoder (reference modules/rel_transformer.py):
// windowed-relative-position self-attention (:137-177), channel LayerNorm (:24-42) and the per-layer condition add
// (:292-295).  Layout: the reference's own [B, C, T] fp32, time contiguous.  The 1x1 / k9 convolutions around them run
// on conv_f32_kernel.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace vsg {

// x = (x + g) * mask, in place (RelativeEncoder.forward :293-295, before the first layer; later layers get it fused into
// the preceding LayerNorm).  g: per-utterance vector [B, C] (g_t == 0) or per-frame tensor [B, C, T] (g_t != 0), or null.
__global__ void relenc_addg_mask_kernel(float* __restrict__ x, const float* __restrict__ g, int g_t,
                                        const float* __restrict__ mask, int C, int T, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int t = (int)(i % T);
  const long long bc = i / T;
  const long long b = bc / C;
  float v = x[i];
  if (g) v += g_t ? g[i] : g[bc];
  x[i] = v * mask[b * T + t];
}

// Channel LayerNorm of [B, C, T] (rel_transformer.py:24-42: mean and biased variance over dim 1, eps inside the rsqrt),
// in place, one thread per (b, t) column (consecutive threads = consecutive t: every channel row is read coalesced),
// followed by what the encoder does next with the result: `x = x + g` (next layer's condition, :293) and `x * x_mask`
// (:295 / :318).  Padded columns only ever feed masked keys and zeroed conv inputs, so storing them as zeros is exact
// for every valid column.
__global__ void relenc_layernorm_kernel(float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                                        const float* __restrict__ g, int g_t, const float* __restrict__ mask, float eps,
                                        int C, int T, int B) {
  const long long col = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= (long long)B * T) return;
  const int b = (int)(col / T), t = (int)(col % T);
  float* xp = x + (long long)b * C * T + t;
  float s = 0.f;
  for (int c = 0; c < C; ++c) s += xp[(long long)c * T];
  const float mean = s / (float)C;
  float v = 0.f;
  for (int c = 0; c < C; ++c) {
    const float d = xp[(long long)c * T] - mean;
    v = fmaf(d, d, v);
  }
  const float rstd = rsqrtf(v / (float)C + eps);
  const float mk = mask[(long long)b * T + t];
  for (int c = 0; c < C; ++c) {
    float y = (xp[(long long)c * T] - mean) * rstd * gamma[c] + beta[c];
    if (g) y += g_t ? g[((long long)b * C + c) * T + t] : g[(long long)b * C + c];
    xp[(long long)c * T] = y * mk;
  }
}

// Self-attention with windowed relative-position keys / values (MultiHeadAttention.attention, rel_transformer.py:137-177):
//   s_ij = (q_i . k_j + [|j-i| <= w] q_i . Ek[j-i+w]) / sqrt(dk);  s_ij = -1e4 where mask_i * mask_j == 0
//   p = softmax_j(s);  o_i = sum_j p_ij (v_j + [|j-i| <= w] Ev[j-i+w])
// qkv: [B, 3 * n_heads * dk, T] (q rows, then k rows, then v rows; head h owns rows h*dk ..); o: [B, n_heads * dk, T];
// Ek / Ev: [2w+1][dk] (heads_share = True).  One CTA = 64 queries of one (utterance, head), 256 threads as a 16 x 16 grid
// of 4 x 4 score sub-tiles; keys stream in tiles of 64 with an online softmax (flash-attention style, fp32 throughout).
constexpr int kAttTile = 64;

template <int DK>
__global__ void __launch_bounds__(256) relenc_attention_f32_kernel(const float* __restrict__ qkv, const float* __restrict__ mask,
                                                                   const float* __restrict__ Ek, const float* __restrict__ Ev,
                                                                   float* __restrict__ o, int n_heads, int T, int w) {
  constexpr int NT = kAttTile, VS = NT + 1, DPT = DK / 16;      // DPT: output dims per thread
  extern __shared__ float sm[];
  float* Qs = sm;                     // [DK][NT]   (d-major; reused to stage the output)
  float* Ks = Qs + DK * NT;           // [DK][NT]
  float* Vs = Ks + DK * NT;           // [DK][VS]
  float* Ps = Vs + DK * VS;           // [NT][VS]
  float* Eks = Ps + NT * VS;          // [2w+1][DK]
  float* Evs = Eks + (2 * w + 1) * DK;
  float* Rq = Evs + (2 * w + 1) * DK; // [NT][2w+1]  q_i . Ek[m]
  float* mq = Rq + NT * (2 * w + 1);  // [NT] query mask
  float* mk = mq + NT;                // [NT] key mask
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * NT;
  const int H = n_heads * DK, nrel = 2 * w + 1;
  const float* qb = qkv + ((long long)b * 3 * H + h * DK) * T;
  const float* kb = qb + (long long)H * T;
  const float* vb = kb + (long long)H * T;
  const float* mb = mask + (long long)b * T;
  const float scale = rsqrtf((float)DK);

  for (int i = tid; i < DK * NT; i += 256) {
    const int d = i / NT, t = q0 + (i % NT);
    Qs[i] = t < T ? qb[(long long)d * T + t] : 0.f;
  }
  for (int i = tid; i < nrel * DK; i += 256) { Eks[i] = Ek[i]; Evs[i] = Ev[i]; }
  if (tid < NT) mq[tid] = (q0 + tid < T) ? mb[q0 + tid] : 0.f;
  __syncthreads();
  for (int i = tid; i < NT * nrel; i += 256) {
    const int r = i / nrel, m = i % nrel;
    float s = 0.f;
    for (int d = 0; d < DK; ++d) s = fmaf(Qs[d * NT + r], Eks[m * DK + d], s);
    Rq[i] = s;
  }

  float row_max[4], row_sum[4], acc[4][DPT];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    row_max[r] = -INFINITY; row_sum[r] = 0.f;
#pragma unroll
    for (int m = 0; m < DPT; ++m) acc[r][m] = 0.f;
  }

  for (int k0 = 0; k0 < T; k0 += NT) {
    __syncthreads();                                  // previous tile's Ks / Vs / Ps fully consumed (and Rq written)
    for (int i = tid; i < DK * NT; i += 256) {
      const int d = i / NT, jj = i % NT, t = k0 + jj;
      const bool ok = t < T;
      Ks[i] = ok ? kb[(long long)d * T + t] : 0.f;
      Vs[d * VS + jj] = ok ? vb[(long long)d * T + t] : 0.f;
    }
    if (tid < NT) mk[tid] = (k0 + tid < T) ? mb[k0 + tid] : 0.f;
    __syncthreads();
    // ---- scores of my 4 x 4 sub-tile
    float s[4][4];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) s[r][c] = 0.f;
#pragma unroll 4
    for (int d = 0; d < DK; ++d) {
      const float4 qv = *reinterpret_cast<const float4*>(Qs + d * NT + ty * 4);
      const float4 kv = *reinterpret_cast<const float4*>(Ks + d * NT + tx * 4);
      const float qa[4] = {qv.x, qv.y, qv.z, qv.w}, ka[4] = {kv.x, kv.y, kv.z, kv.w};
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) s[r][c] = fmaf(qa[r], ka[c], s[r][c]);
    }
    float tile_max[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int i = ty * 4 + r, qi = q0 + i;
      tile_max[r] = -INFINITY;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int j = tx * 4 + c, kj = k0 + j;
        float v = s[r][c];
        const int rel = kj - qi + w;
        if (rel >= 0 && rel < nrel) v += Rq[i * nrel + rel];
        v *= scale;
        if (mq[i] * mk[j] == 0.f) v = -1e4f;
        if (kj >= T) v = -INFINITY;                   // beyond the sequence: not a key at all
        s[r][c] = v;
        tile_max[r] = fmaxf(tile_max[r], v);
      }
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) tile_max[r] = fmaxf(tile_max[r], __shfl_xor_sync(0xffffffffu, tile_max[r], off));
    }
    // ---- online softmax: rescale the running sums, publish the un-normalised probabilities
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const float new_max = fmaxf(row_max[r], tile_max[r]);
      const float corr = expf(row_max[r] - new_max);            // 0 for the first tile (row_max = -inf)
      row_max[r] = new_max;
      float psum = 0.f;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const float pv = expf(s[r][c] - new_max);
        Ps[(ty * 4 + r) * VS + tx * 4 + c] = pv;
        psum += pv;
      }
#pragma unroll
      for (int off = 8; off > 0; off >>= 1) psum += __shfl_xor_sync(0xffffffffu, psum, off);
      row_sum[r] = row_sum[r] * corr + psum;
#pragma unroll
      for (int m = 0; m < DPT; ++m) acc[r][m] *= corr;
    }
    __syncthreads();
    // ---- o += P V (+ relative-position values on the 2w+1 diagonals)
    for (int j = 0; j < NT; ++j) {
      float vv[DPT];
#pragma unroll
      for (int m = 0; m < DPT; ++m) vv[m] = Vs[(tx + 16 * m) * VS + j];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const float pv = Ps[(ty * 4 + r) * VS + j];
#pragma unroll
        for (int m = 0; m < DPT; ++m) acc[r][m] = fmaf(pv, vv[m], acc[r][m]);
      }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int i = ty * 4 + r, qi = q0 + i;
      for (int rel = 0; rel < nrel; ++rel) {
        const int j = qi + rel - w - k0;              // key position inside this tile
        if (j < 0 || j >= NT || k0 + j >= T) continue;
        const float pv = Ps[i * VS + j];
#pragma unroll
        for (int m = 0; m < DPT; ++m) acc[r][m] = fmaf(pv, Evs[rel * DK + tx + 16 * m], acc[r][m]);
      }
    }
  }
  // ---- normalise, stage [d][i] in Qs, write coalesced
  __syncthreads();
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const float inv = 1.0f / row_sum[r];
#pragma unroll
    for (int m = 0; m < DPT; ++m) Qs[(tx + 16 * m) * NT + ty * 4 + r] = acc[r][m] * inv;
  }
  __syncthreads();
  float* ob = o + ((long long)b * H + h * DK) * T;
  for (int i = tid; i < DK * NT; i += 256) {
    const int d = i / NT, t = q0 + (i % NT);
    if (t < T) ob[(long long)d * T + t] = Qs[i];
  }
}

// Length regulator + positional embedding (SURVEY.md section 8 row f2), one CTA per utterance:
//   y[b, :, t] = enc[b, :, mel2ph[b, t] - 1]   (0 where mel2ph == 0)      expand_states, models/commons/align_ops.py:22-26
//   keep_t = (y[b, 0, t] != 0);  pos_t = cumsum(keep)_t * keep_t            make_positions, modules/rel_transformer.py:78-88
//   y[b, :, t] += table[pos_t, :]                                           models/visinger.py:79-82 (table row 0 is zero)
// -- the position of a frame is the running count of frames whose channel 0 is non-zero, the reference's data-dependent
// definition.  enc: [B, H, T_ph]; mel2ph: int64 [B, T]; table: [rows, H] (SinusoidalPositionalEmbedding.weights) or null.
// The utterance is processed in chunks of kLrChunk frames (token indices, scan with the carry of the chunks before, then
// the chunk's y), so shared memory does not depend on T.  Launch with kLrThreads threads.
constexpr int kLrThreads = 512, kLrChunk = 2048;
__global__ void __launch_bounds__(kLrThreads) length_regulate_pos_kernel(const float* __restrict__ enc,
                                                                         const long long* __restrict__ mel2ph,
                                                                         const float* __restrict__ table, int table_rows,
                                                                         float* __restrict__ y, int H, int T_ph, int T) {
  __shared__ int tok[kLrChunk];                  // token index of each frame of the chunk (-1 = padding)
  __shared__ int pos[kLrChunk];                  // its position
  __shared__ int warp_tot[kLrThreads / 32];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = kLrThreads / 32;
  const float* eb = enc + (long long)b * H * T_ph;
  float* yb = y + (long long)b * H * T;
  int carry = 0;                                 // frames kept before this chunk
  for (int c0 = 0; c0 < T; c0 += kLrChunk) {
    const int n = min(kLrChunk, T - c0);
    for (int t = tid; t < n; t += kLrThreads) {
      const long long m = mel2ph[(long long)b * T + c0 + t];
      tok[t] = (m > 0 && m <= T_ph) ? (int)(m - 1) : -1;
    }
    __syncthreads();
    // inclusive scan of keep_t, kLrThreads frames at a time
    for (int t0 = 0; t0 < n; t0 += kLrThreads) {
      const int t = t0 + tid;
      int keep = 0;
      if (t < n && tok[t] >= 0) keep = (eb[tok[t]] != 0.f) ? 1 : 0;           // channel 0 of the gathered row
      int v = keep;
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const int x = __shfl_up_sync(0xffffffffu, v, off);
        if (lane >= off) v += x;
      }
      if (lane == 31) warp_tot[warp] = v;
      __syncthreads();
      int before = carry;
      for (int wv = 0; wv < warp; ++wv) before += warp_tot[wv];
      if (t < n) pos[t] = keep ? before + v : 0;
      int part = 0;
      for (int wv = 0; wv < nw; ++wv) part += warp_tot[wv];
      carry += part;
      __syncthreads();
    }
    for (int i = tid; i < H * n; i += kLrThreads) {
      const int c = i / n, t = i - c * n;
      float v = tok[t] >= 0 ? eb[(long long)c * T_ph + tok[t]] : 0.f;
      if (table && pos[t] < table_rows) v += table[(long long)pos[t] * H + c];
      yb[(long long)c * T + c0 + t] = v;
    }
    __syncthreads();                             // tok / pos are rewritten by the next chunk
  }
}

// FramePriorNetwork head + prior sampling (SURVEY.md section 8 row f2), fp32 layout:
//   stats = proj(h) * mask  (Conv1d(H -> 2H, 1), modules/visinger/encoder.py:65,71);  (mu_p, logs_p) = split(stats)  (:72)
//   z_p = (mu_p + noise * exp(logs_p)) * mask                                              models/visinger.py:107
// One thread owns one (channel, frame): both dot products of length H, the sample, three stores (stats may be null).
// W: [2H][H] row-major; h, noise, z: [B, H, T]; stats: [B, 2H, T].
__global__ void prior_head_f32_kernel(const float* __restrict__ h, const float* __restrict__ W, const float* __restrict__ bias,
                                      const float* __restrict__ noise, const float* __restrict__ mask, float* __restrict__ stats,
                                      float* __restrict__ z, int H, int T) {
  extern __shared__ float ph_sm[];              // [H][32] frames of h
  const int b = blockIdx.y, t0 = blockIdx.x * 32, tx = threadIdx.x & 31, ty = threadIdx.x >> 5, nty = blockDim.x >> 5;
  const int t = t0 + tx;
  for (int c = ty; c < H; c += nty) ph_sm[c * 32 + tx] = t < T ? h[((long long)b * H + c) * T + t] : 0.f;
  __syncthreads();
  if (t >= T) return;
  const float mk = mask[(long long)b * T + t];
  for (int c = ty; c < H; c += nty) {
    float mu = bias[c], lg = bias[H + c];
    const float* wm = W + (long long)c * H;
    const float* wl = W + (long long)(H + c) * H;
    for (int k = 0; k < H; ++k) {
      const float hv = ph_sm[k * 32 + tx];
      mu = fmaf(wm[k], hv, mu);
      lg = fmaf(wl[k], hv, lg);
    }
    mu *= mk; lg *= mk;
    const long long o = ((long long)b * H + c) * T + t;
    if (stats) {
      stats[((long long)b * 2 * H + c) * T + t] = mu;
      stats[((long long)b * 2 * H + H + c) * T + t] = lg;
    }
    z[o] = (mu + noise[o] * expf(lg)) * mk;
  }
}

inline size_t relenc_attention_f32_smem(int dk, int w) {
  const int NT = kAttTile, VS = NT + 1, nrel = 2 * w + 1;
  return sizeof(float) * ((size_t)2 * dk * NT + (size_t)dk * VS + (size_t)NT * VS + (size_t)2 * nrel * dk + (size_t)NT * nrel + 2 * NT);
}

}  // namespace vsg
