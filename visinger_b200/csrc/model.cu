// The whole model in one call (vsg_model_pack_create / vsg_model_forward): the token-rate glue of VISinger.forward as
// fp32 CUDA-core kernels, chained with the existing stacks (RelativeEncoder, length regulator, frame-prior head, flow and
// decoder).  Also the seeded prior noise (vsg_normal_noise) and the sinusoidal position table.  Voice conversion
// (vsg_convert_pack_create / vsg_spectrogram / vsg_model_convert): waveform -> linear spectrogram -> posterior encoder ->
// flow forward -> flow reverse -> decoder, with the DFT basis of the spectrogram packed here.
#include "vsg_common.cuh"
#include "run.cuh"
#include "pack_tc.cuh"

#include <math.h>

namespace vsg {

namespace {

// ---- kernels --------------------------------------------------------------------------------------------------------

// frame mask [B, T] = (mel2ph > 0) , then the sinusoidal table [rows, dim]
// (SinusoidalPositionalEmbedding.get_embedding, modules/rel_transformer.py:46-55, padding_idx 0): one grid over both.
// a = fp32(p) * freq[k] rounded to fp32 as torch does; sin / cos in double, rounded once.  freq null: the correctly
// rounded exp of the same fp32 exponent k * fp32(-ln(10000) / (half - 1)).
__global__ void model_prep_kernel(const long long* __restrict__ mel2ph, float* __restrict__ mask, long long n_mask,
                                  const float* __restrict__ freq, float step, float* __restrict__ table, int rows, int dim) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_mask) {
    mask[i] = mel2ph[i] > 0 ? 1.f : 0.f;
    return;
  }
  const long long j = i - n_mask;
  if (!table || j >= (long long)rows * dim) return;
  const int p = (int)(j / dim), c = (int)(j - (long long)p * dim), half = dim / 2;
  float v = 0.f;
  if (p > 0 && c < 2 * half) {
    const int k = c < half ? c : c - half;
    const float f = freq ? freq[k] : (float)exp((double)__fmul_rn((float)k, step));
    const float a = __fmul_rn((float)p, f);
    v = c < half ? (float)sin((double)a) : (float)cos((double)a);
  }
  table[j] = v;
}

// TextEncoder.encode_tokens up to the positions (modules/visinger/encoder.py:57-61):
//   x = cat(ph_emb[text], pitch_emb[pitch], dur_emb[dur]) * fp32(sqrt(H));  y = (Linear(3H -> H)(x)) * (text > 0)
// kFeTok tokens per CTA share every weight load; the weight is stored transposed [3H][H] so a warp's loads are
// contiguous.  fp32 FFMA accumulation in input order, then + bias.  Writes y as [B, H, T_ph] (the encoder's layout) and
// the token mask [B, T_ph].
constexpr int kFeTok = 8;
__global__ void __launch_bounds__(256) token_frontend_kernel(
    const long long* __restrict__ text, const long long* __restrict__ pitch, const long long* __restrict__ dur,
    const float* __restrict__ ph_emb, int n_ph, const float* __restrict__ pitch_emb, int n_pitch,
    const float* __restrict__ dur_emb, int n_dur, const float* __restrict__ wt, const float* __restrict__ bias, float scale,
    float* __restrict__ y, float* __restrict__ tokmask, int H, int T_ph, long long n_tok) {
  extern __shared__ float xs[];                  // [kFeTok][3H]
  __shared__ float nonpad[kFeTok];
  const long long tok0 = (long long)blockIdx.x * kFeTok;
  const int K = 3 * H;
  for (int i = threadIdx.x; i < kFeTok * K; i += blockDim.x) {
    const int tt = i / K, k = i - tt * K, s = k / H, c = k - s * H;
    const long long tok = tok0 + tt;
    float v = 0.f;
    if (tok < n_tok) {
      const long long id = (s == 0 ? text : s == 1 ? pitch : dur)[tok];
      const int n = s == 0 ? n_ph : s == 1 ? n_pitch : n_dur;
      const float* tab = s == 0 ? ph_emb : s == 1 ? pitch_emb : dur_emb;
      if (id >= 0 && id < n) v = __fmul_rn(tab[id * H + c], scale);
    }
    xs[i] = v;
  }
  if (threadIdx.x < kFeTok) {
    const long long tok = tok0 + threadIdx.x;
    const float np = (tok < n_tok && text[tok] > 0) ? 1.f : 0.f;
    nonpad[threadIdx.x] = np;
    if (tok < n_tok) tokmask[tok] = np;
  }
  __syncthreads();
  for (int o = threadIdx.x; o < H; o += blockDim.x) {
    float acc[kFeTok];
#pragma unroll
    for (int tt = 0; tt < kFeTok; ++tt) acc[tt] = 0.f;
    for (int k = 0; k < K; ++k) {
      const float w = wt[(long long)k * H + o];
#pragma unroll
      for (int tt = 0; tt < kFeTok; ++tt) acc[tt] = fmaf(xs[tt * K + k], w, acc[tt]);
    }
#pragma unroll
    for (int tt = 0; tt < kFeTok; ++tt) {
      const long long tok = tok0 + tt;
      if (tok >= n_tok) break;
      const long long b = tok / T_ph, t = tok - b * T_ph;
      y[(b * H + o) * T_ph + t] = __fmul_rn(__fadd_rn(acc[tt], bias[o]), nonpad[tt]);
    }
  }
}

// The reference's positional term of the text encoder, bit for bit (modules/visinger/encoder.py:50-53): it calls
// SinusoidalPositionalEmbedding with seq_len = H, so the [T_ph, H] lookup of one utterance is *viewed* as [H, T_ph] and
// transposed back.  In the [H, T_ph] layout of y that view is the identity on flat indices: element e of utterance b
// gains table[pos[e / H], e % H], where pos_t = running count of tokens whose channel 0 is non-zero (0 on the others).
// Then the mask again.  One CTA per utterance: the scan of channel 0, then the in-place update.
constexpr int kPosThreads = 1024;
__global__ void __launch_bounds__(kPosThreads) token_positions_kernel(float* __restrict__ y, const float* __restrict__ tokmask,
                                                                      const float* __restrict__ table, int* __restrict__ posbuf,
                                                                      int H, int T_ph) {
  __shared__ int warp_tot[kPosThreads / 32];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = kPosThreads / 32;
  float* yb = y + (long long)b * H * T_ph;
  int* pos = posbuf + (long long)b * T_ph;
  int carry = 0;
  for (int t0 = 0; t0 < T_ph; t0 += kPosThreads) {
    const int t = t0 + tid;
    const int keep = (t < T_ph && yb[t] != 0.f) ? 1 : 0;     // channel 0 of token t
    int v = keep;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const int x = __shfl_up_sync(0xffffffffu, v, off);
      if (lane >= off) v += x;
    }
    if (lane == 31) warp_tot[warp] = v;
    __syncthreads();
    int before = carry, part = 0;
    for (int wv = 0; wv < nw; ++wv) {
      if (wv < warp) before += warp_tot[wv];
      part += warp_tot[wv];
    }
    if (t < T_ph) pos[t] = keep ? before + v : 0;
    carry += part;
    __syncthreads();
  }
  const float* mb = tokmask + (long long)b * T_ph;
  const long long n = (long long)H * T_ph;
  for (long long e = tid; e < n; e += kPosThreads) {
    const long long r = e / H;
    const int c = (int)(e - r * H);
    yb[e] = __fmul_rn(__fadd_rn(yb[e], table[(long long)pos[r] * H + c]), mb[e % T_ph]);
  }
}

// VISinger.speaker_embedding, summed in its order: spk_embed_proj(spk_embed) (Linear, fp32),
// then + spk_id_proj[spk_id].  One warp per (utterance, channel); ids of up to kSpkChunk utterances per launch travel as
// a kernel argument (they are host data, range-checked before any launch).
constexpr int kSpkChunk = 64;
struct SpkIds { int32_t id[kSpkChunk]; };
__global__ void speaker_cond_kernel(const float* __restrict__ We, const float* __restrict__ be, const float* __restrict__ emb,
                                    int E, const float* __restrict__ id_table, SpkIds ids, int b0, int nb,
                                    float* __restrict__ g, int gin) {
  const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (gw >= nb * gin) return;
  const int bl = gw / gin, o = gw - bl * gin, b = b0 + bl;
  float s = 0.f;
  if (We) {
    const float* wr = We + (long long)o * E;
    const float* er = emb + (long long)b * E;
    for (int i = lane; i < E; i += 32) s = fmaf(wr[i], er[i], s);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    s = __fadd_rn(s, be[o]);
  }
  if (id_table) s = __fadd_rn(s, id_table[(long long)ids.id[bl] * gin + o]);
  if (lane == 0) g[(long long)b * gin + o] = s;
}

// PitchPredictor.linear (Conv1d(H -> 2, 1)) and VISinger.forward_pitch:
// pred [B, T, 2]; cond [B, 1, T] = (f0 * voiced) * mask with f0 = pred[..., 0],
// voiced = pred[..., 1] <= 0, or f0 / uv given: voiced = uv == 0.  One thread per frame.
__global__ void pitch_head_kernel(const float* __restrict__ h, const float* __restrict__ w, const float* __restrict__ bias,
                                  const float* __restrict__ f0, const float* __restrict__ uv, const float* __restrict__ mask,
                                  float* __restrict__ pred, float* __restrict__ cond, int H, int T, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long b = i / T, t = i - b * T;
  const float* hb = h + b * H * T + t;
  float a0 = 0.f, a1 = 0.f;
  for (int c = 0; c < H; ++c) {
    const float v = hb[(long long)c * T];
    a0 = fmaf(w[c], v, a0);
    a1 = fmaf(w[H + c], v, a1);
  }
  const float p0 = __fadd_rn(a0, bias[0]), p1 = __fadd_rn(a1, bias[1]);
  pred[2 * i] = p0;
  pred[2 * i + 1] = p1;
  const float fv = f0 ? f0[i] : p0;
  const float voiced = f0 ? (uv[i] == 0.f ? 1.f : 0.f) : (p1 <= 0.f ? 1.f : 0.f);
  cond[i] = __fmul_rn(__fmul_rn(fv, voiced), mask[i]);
}

// Philox4x32-10 (Salmon et al., SC'11), one 128-bit block per element.
__device__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
    const uint32_t lo0 = 0xD2511F53u * c[0], hi0 = __umulhi(0xD2511F53u, c[0]);
    const uint32_t lo1 = 0xCD9E8D57u * c[2], hi1 = __umulhi(0xCD9E8D57u, c[2]);
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
    c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
  }
}

// out [B, C, T] holds frames [t_base, t_base + T) of the noise: element (b, c, t) draws counter (t_base + t, c)
__global__ void normal_noise_kernel(const unsigned long long* __restrict__ seeds, float* __restrict__ out, int C, int T,
                                    long long n, int t_base) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long CT = (long long)C * T, b = i / CT, r = i - b * CT;
  const uint32_t c = (uint32_t)(r / T), t = (uint32_t)(r - (long long)c * T);
  const unsigned long long s = seeds[b];
  uint32_t x[4] = {(uint32_t)t_base + t, c, 0u, 0u};
  philox4x32_10(x, (uint32_t)s, (uint32_t)(s >> 32));
  const double u1 = ((double)x[0] + 1.0) * 2.3283064365386963e-10, u2 = (double)x[1] * 2.3283064365386963e-10;
  out[i] = (float)(sqrt(-2.0 * log(u1)) * cos(6.283185307179586 * u2));
}

// ---- launchers ------------------------------------------------------------------------------------------------------

float freq_step(int dim) { return (float)(-(log(10000.0) / (dim / 2 - 1))); }

int launch_prep(const long long* mel2ph, float* mask, long long n_mask, const float* freq, float* table, int rows, int dim,
                cudaStream_t st) {
  const long long n = n_mask + (table ? (long long)rows * dim : 0);
  if (n == 0) return VSG_OK;
  model_prep_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(mel2ph, mask, n_mask, freq, dim >= 4 ? freq_step(dim) : 0.f,
                                                                 table, rows, dim);
  VSG_LAUNCH_CHECK("model_prep_kernel");
  return VSG_OK;
}

int launch_noise(const uint64_t* seeds, float* out, int B, int C, int T, cudaStream_t st, int t_base = 0) {
  const long long n = (long long)B * C * T;
  normal_noise_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const unsigned long long*)seeds, out, C, T, n, t_base);
  VSG_LAUNCH_CHECK("normal_noise_kernel");
  return VSG_OK;
}

bool relenc_bf16(int precision) { return precision == VSG_PRECISION_BF16; }

int relenc_run(const VsgPack* P, const float* x, const float* mask, const float* g, float* y, int B, int T, int precision,
               Workspace& ws, cudaStream_t st) {
  const size_t mark = ws.off;
  const int rc = relenc_bf16(precision) ? relenc_forward_tc(P, x, mask, g, 0, y, B, T, ws, st)
                                        : relenc_forward_f32(P, x, mask, g, 0, y, B, T, ws, st);
  ws.off = mark;
  return rc;
}

size_t relenc_ws(const VsgPack* P, int B, int T, int precision) {
  return relenc_bf16(precision) ? relenc_ws_bytes_tc(P, B, T, 0) : relenc_ws_bytes_f32(P, B, T, 0);
}

size_t model_ws_bytes(const VsgPack* P, int B, int T_ph, int T, int precision) {
  const ModelPack& m = *P->model;
  const size_t H = m.cfg.hidden, rows = (size_t)std::max(T, T_ph) + 1, BT = (size_t)B * T;
  const int rp = relenc_bf16(precision) ? VSG_PRECISION_BF16 : VSG_PRECISION_FP32;
  const size_t persist = align256(BT * 4) + align256((size_t)B * T_ph * 4) + align256((size_t)B * m.gin * 4) +
                         align256(BT * H * 4);
  size_t p1 = align256(rows * H * 4) + align256((size_t)B * H * T_ph * 4) +
              align256((size_t)B * T_ph * 4) + 3 * align256(BT * H * 4) + align256(BT * 4) + align256(BT * 2 * 4);
  size_t sub = std::max(relenc_ws(m.text, B, T_ph, rp), frame_prior_ws_bytes(m.prior, B, T, rp));
  if (m.cfg.use_pitch_embed) sub = std::max(sub, relenc_ws(m.pitch, B, T, rp));
  const size_t hot = vsg_workspace_bytes(m.hot, B, T, precision);
  return persist + std::max(p1 + sub, hot) + 4096;
}

// g [B, gin] = VISinger.speaker_embedding for host ids spk_id (range-checked by the caller) and device spk_embed
int speaker_cond(const ModelPack& m, const int64_t* spk_id, const float* spk_embed, float* g, int B, cudaStream_t st) {
  const VsgModelConfig& c = m.cfg;
  const int gin = m.gin;
  for (int b0 = 0; b0 < B; b0 += kSpkChunk) {
    const int nb = std::min(kSpkChunk, B - b0);
    SpkIds ids;
    for (int i = 0; i < kSpkChunk; ++i) ids.id[i] = (spk_id && i < nb) ? (int32_t)spk_id[b0 + i] : 0;
    const long long threads = (long long)nb * gin * 32;
    speaker_cond_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(
        c.use_spk_embed ? m.spk_embed_w : nullptr, m.spk_embed_b, spk_embed, c.spk_embed_dim,
        c.use_spk_id ? m.spk_id_w : nullptr, ids, b0, nb, g, gin);
    VSG_LAUNCH_CHECK("speaker_cond_kernel");
  }
  return VSG_OK;
}

// VISinger.forward(infer=True), after validation.
int model_forward(const VsgPack* P, const long long* text, const long long* pitch, const long long* dur,
                  const long long* mel2ph, const int64_t* spk_id, const float* spk_embed, const float* f0, const float* uv,
                  const float* noise, const uint64_t* seeds, float* wav, float* f0_pred, float* z_q_out, int B, int T_ph,
                  int T, int precision, Workspace& ws, cudaStream_t st) {
  const ModelPack& m = *P->model;
  const VsgModelConfig& c = m.cfg;
  const int H = c.hidden, gin = m.gin, rows = std::max(T, T_ph) + 1;
  const size_t BT = (size_t)B * T;
  // live for the whole call
  float* mask = ws.take<float>(BT);
  float* tokmask = ws.take<float>((size_t)B * T_ph);
  float* g = ws.take<float>((size_t)B * gin);
  float* z_p = ws.take<float>(BT * H);
  const size_t mark0 = ws.off;
  // live until the frame prior has run; the flow and decoder reuse all of it
  float* table = ws.take<float>((size_t)rows * H);
  float* tok = ws.take<float>((size_t)B * H * T_ph);
  int* posbuf = ws.take<int>((size_t)B * T_ph);
  float* x = ws.take<float>(BT * H);         // prior input: length-regulated tokens + frame positions
  float* hp = ws.take<float>(BT * H);        // pitch predictor output
  float* nz = ws.take<float>(BT * H);        // drawn noise
  float* cond = ws.take<float>(BT);
  float* pred = f0_pred ? f0_pred : ws.take<float>(BT * 2);
  if (ws.overflow) return fail(VSG_ENOMEM, "model workspace too small: need %zu bytes", ws.off);

  VSG_TRY(launch_prep(mel2ph, mask, (long long)BT, m.freq, table, rows, H, st));
  {  // TextEncoder.encode_tokens (modules/visinger/encoder.py:57-68)
    const long long n_tok = (long long)B * T_ph;
    const size_t sm = (size_t)kFeTok * 3 * H * sizeof(float);
    if (sm > 48 * 1024)
      VSG_CUDA_TRY(cudaFuncSetAttribute(token_frontend_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    token_frontend_kernel<<<(unsigned)((n_tok + kFeTok - 1) / kFeTok), 256, sm, st>>>(
        text, pitch, dur, m.ph_emb, c.ph_dict_size, m.pitch_emb, c.pitch_size, m.dur_emb, c.dur_size, m.lin_wt, m.lin_b,
        (float)sqrt((double)H), tok, tokmask, H, T_ph, n_tok);
    VSG_LAUNCH_CHECK("token_frontend_kernel");
    // always: VISinger builds its TextEncoder with use_pos_embed=True; the hparam governs the frame positions below
    token_positions_kernel<<<B, kPosThreads, 0, st>>>(tok, tokmask, table, posbuf, H, T_ph);
    VSG_LAUNCH_CHECK("token_positions_kernel");
    VSG_TRY(relenc_run(m.text, tok, tokmask, nullptr, tok, B, T_ph, precision, ws, st));
  }
  // length regulator + frame positions
  VSG_TRY(length_regulate(tok, mel2ph, c.use_pos_embed ? table : nullptr, c.use_pos_embed ? rows : 0, x, B, H, T_ph, T, st));
  // speaker condition [B, gin, 1]
  VSG_TRY(speaker_cond(m, spk_id, spk_embed, g, B, st));
  if (c.use_pitch_embed) {   // VISinger.forward_pitch
    VSG_TRY(relenc_run(m.pitch, x, mask, g, hp, B, T, precision, ws, st));
    pitch_head_kernel<<<(unsigned)((BT + 255) / 256), 256, 0, st>>>(hp, m.pitch_w, m.pitch_b, f0, uv, mask, pred, cond, H, T,
                                                                    (long long)BT);
    VSG_LAUNCH_CHECK("pitch_head_kernel");
  }
  if (!noise) {
    VSG_TRY(launch_noise(seeds, nz, B, H, T, st));
    noise = nz;
  }
  {  // frame prior network + proj + prior sampling (models/visinger.py:86-107)
    const size_t mark = ws.off;
    const float* gc = c.use_pitch_embed ? cond : nullptr;
    if (relenc_bf16(precision)) VSG_TRY(frame_prior_forward_tc(m.prior, x, mask, gc, noise, nullptr, z_p, B, T, ws, st));
    else VSG_TRY(frame_prior_forward_f32(m.prior, x, mask, gc, noise, nullptr, z_p, B, T, ws, st));
    ws.off = mark;
  }
  // flow reverse + decoder (models/visinger.py:109-111)
  ws.off = mark0;
  return infer_zp_run(m.hot, z_p, mask, g, wav, z_q_out, B, T, precision, ws, st);
}

// ---- voice conversion -----------------------------------------------------------------------------------------------

bool convert_bf16(int precision) { return precision == VSG_PRECISION_BF16; }   // spectrogram + posterior on tcgen05

// what vsg_spectrogram takes: mask, the bf16 spectrogram (tcgen05 path) and the framed rows
size_t spectrogram_ws_bytes(const VsgPack* P, int B, int T, int precision) {
  const ModelPack& m = *P->model;
  const size_t BT = (size_t)B * T;
  const bool bf = convert_bf16(precision);
  return align256(BT * 4) + (bf ? align256(BT * m.post->enc.in_pad * 2) : 0) + spec_frames_bytes(m.spec, B, T, bf) + 256;
}

size_t convert_ws_bytes(const VsgPack* P, int B, int T, int precision) {
  const ModelPack& m = *P->model;
  const EncPack& en = m.post->enc;
  const size_t BT = (size_t)B * T, H = m.cfg.hidden;
  const bool bf = convert_bf16(precision);
  const size_t persist = align256(BT * 4) + 2 * align256((size_t)B * m.gin * 4) + 2 * align256(BT * H * 4);
  const size_t keep = (bf ? align256(BT * en.in_pad * 2) : align256(BT * m.spec.bins * 4)) + align256(BT * H * 4) +
                      align256(BT * 2 * en.out_channels * 4);
  const size_t post = bf ? posterior_ws_bytes_tc(m.post, B, T) : posterior_ws_bytes_f32(m.post, B, T);
  const size_t stage1 = keep + std::max(spec_frames_bytes(m.spec, B, T, bf) + 256, post);
  return persist + std::max(stage1, vsg_workspace_bytes(m.hot, B, T, precision)) + 4096;
}

// vsg_model_convert after validation: exactly one of wav / spec.
int model_convert(const VsgPack* P, const float* wav, const float* spec, const int32_t* lengths, const int64_t* src_id,
                  const float* src_embed, const int64_t* tgt_id, const float* tgt_embed, const float* noise,
                  const uint64_t* seeds, float* wav_out, float* spec_out, float* z_out, int B, int T, int precision,
                  Workspace& ws, cudaStream_t st) {
  const ModelPack& m = *P->model;
  const SpecPack& S = m.spec;
  const EncPack& en = m.post->enc;
  const int H = m.cfg.hidden, gin = m.gin;
  const size_t BT = (size_t)B * T;
  const bool bf = convert_bf16(precision);
  // live for the whole call
  float* mask = ws.take<float>(BT);
  float* g_src = ws.take<float>((size_t)B * gin);
  float* g_tgt = ws.take<float>((size_t)B * gin);
  float* z = ws.take<float>(BT * H);         // posterior sample
  float* z_p = ws.take<float>(BT * H);       // flow(z, g_src)
  const size_t mark0 = ws.off;
  // live until the posterior has run
  __nv_bfloat16* u = (bf && wav) ? ws.take<__nv_bfloat16>(BT * en.in_pad) : nullptr;
  float* x = (!bf && wav) ? (spec_out ? spec_out : ws.take<float>(BT * S.bins)) : nullptr;
  float* nz = noise ? nullptr : ws.take<float>(BT * H);
  float* stats = ws.take<float>(BT * 2 * en.out_channels);
  if (ws.overflow) return fail(VSG_ENOMEM, "convert workspace too small: need %zu bytes", ws.off);

  VSG_TRY(lengths_mask(lengths, mask, B, T, st));
  VSG_TRY(speaker_cond(m, src_id, src_embed, g_src, B, st));
  VSG_TRY(speaker_cond(m, tgt_id, tgt_embed, g_tgt, B, st));
  if (!noise) {
    VSG_TRY(launch_noise(seeds, nz, B, H, T, st));
    noise = nz;
  }
  // z = posterior_encoder(spec, mask, g_src)                       (modules/visinger/encoder.py:92-98)
  if (bf && wav) {
    VSG_TRY(spectrogram_tc(P, S, en.in_pad, wav, lengths, mask, u, B, T, ws, st));
    if (spec_out) VSG_TRY(widen_bf16(u, spec_out, B, S.bins, en.in_pad, T, st));
    VSG_TRY(posterior_core_tc(m.post, u, mask, g_src, noise, z, stats, B, T, ws, st));
  } else if (bf) {
    VSG_TRY(posterior_forward_tc(m.post, spec, mask, g_src, noise, z, stats, B, T, ws, st));
  } else {
    if (wav) {
      const size_t mark = ws.off;
      VSG_TRY(spectrogram_f32(S, wav, lengths, mask, x, B, T, ws, st));
      ws.off = mark;
      spec = x;
    }
    VSG_TRY(posterior_forward_f32(m.post, spec, mask, g_src, noise, z, stats, B, T, ws, st));
  }
  // z_p = flow(z, mask, g_src); then flow(z_p, mask, g_tgt, reverse) * mask and the decoder under g_tgt
  ws.off = mark0;
  VSG_TRY(run_flow(m.hot, z, mask, g_src, z_p, B, T, 0, precision, ws, st));
  ws.off = mark0;
  return infer_zp_run(m.hot, z_p, mask, g_tgt, wav_out, z_out, B, T, precision, ws, st);
}

// ---- voice conversion over a window of frames -----------------------------------------------------------------------
// Frames [t0, t1) of model_convert(wav): every part is convolutional, so the ranges of window_ranges nest outward from
// the decoder's -- flow reverse +-Cf, flow forward +-2 Cf, spectrogram and posterior +-(2 Cf + Cp) -- and each part
// runs over its range with the one pass's kernels (the tcgen05 sums do not depend on tile or row position, the FFMA
// kernels choose nothing by length, the decoder's choices come from (B, T): DESIGN.md 4.8, 4.9).

int post_context(const ModelPack& m) {
  const EncPack& en = m.post->enc;
  return wavenet_context(en.kernel, en.dil_rate, en.n_layers);
}

size_t convert_window_ws_bytes(const VsgPack* P, int B, int T, int n, int precision) {
  const ModelPack& m = *P->model;
  const VsgPack* hot = m.hot;
  const EncPack& en = m.post->enc;
  const int Wd = window_span(hot, B, T, n, precision);
  if (!Wd) return 0;
  const int Wg = std::min(T, Wd + 4 * flow_context(hot)), Wp = std::min(T, Wg + 2 * post_context(m));
  const size_t BP = (size_t)B * Wp, BG = (size_t)B * Wg, H = m.cfg.hidden;
  const bool bf = convert_bf16(precision);
  const size_t persist = align256(BP * 4) + align256(BG * 4) + 2 * align256((size_t)B * m.gin * 4) + align256(BP * H * 4) +
                         align256(BG * H * 4);
  const size_t keep = (bf ? align256(BP * en.in_pad * 2) : align256(BP * m.spec.bins * 4)) + align256(BP * H * 4) +
                      align256(BP * 2 * en.out_channels * 4);
  const size_t post = bf ? posterior_ws_bytes_tc(m.post, B, Wp) : posterior_ws_bytes_f32(m.post, B, Wp);
  const size_t stage1 = keep + std::max(spec_frames_bytes(m.spec, B, Wp, bf) + 256, post);
  const size_t rest = std::max(flow_ws(hot, B, Wg, precision), window_ws(hot, B, T, n, precision));
  return persist + std::max(stage1, rest) + 4096;
}

int model_convert_window(const VsgPack* P, const float* wav, const int32_t* lengths, const int64_t* src_id,
                         const float* src_embed, const int64_t* tgt_id, const float* tgt_embed, const float* noise,
                         const uint64_t* seeds, float* wav_out, int64_t wav_ld, float* z_out, int B, int T, int t0, int t1,
                         int precision, Workspace& ws, cudaStream_t st) {
  const ModelPack& m = *P->model;
  const VsgPack* hot = m.hot;
  const SpecPack& S = m.spec;
  const EncPack& en = m.post->enc;
  const int H = m.cfg.hidden, gin = m.gin;
  WinRange r;
  VSG_TRY(window_ranges(hot, B, T, t0, t1, precision, true, &r, post_context(m)));
  const int Wp = r.pb - r.pa, Wg = r.gb - r.ga;
  const size_t BP = (size_t)B * Wp, BG = (size_t)B * Wg;
  const bool bf = convert_bf16(precision);
  // live for the whole call: the masks of the posterior's and the flow's ranges, the conditions, z and z_p
  float* mask_p = ws.take<float>(BP);
  float* mask_g = ws.take<float>(BG);
  float* g_src = ws.take<float>((size_t)B * gin);
  float* g_tgt = ws.take<float>((size_t)B * gin);
  float* z = ws.take<float>(BP * H);
  float* z_p = ws.take<float>(BG * H);
  const size_t mark0 = ws.off;
  // live until the posterior has run
  __nv_bfloat16* u = bf ? ws.take<__nv_bfloat16>(BP * en.in_pad) : nullptr;
  float* x = bf ? nullptr : ws.take<float>(BP * S.bins);
  float* nz = ws.take<float>(BP * H);
  float* stats = ws.take<float>(BP * 2 * en.out_channels);
  if (ws.overflow) return fail(VSG_ENOMEM, "convert window workspace too small: need %zu bytes", ws.off);

  VSG_TRY(lengths_mask(lengths, mask_p, B, Wp, st, r.pa, T));
  VSG_TRY(lengths_mask(lengths, mask_g, B, Wg, st, r.ga, T));
  VSG_TRY(speaker_cond(m, src_id, src_embed, g_src, B, st));
  VSG_TRY(speaker_cond(m, tgt_id, tgt_embed, g_tgt, B, st));
  if (noise)   // the posterior's range of the caller's [B, H, T] noise
    VSG_CUDA_TRY(cudaMemcpy2DAsync(nz, (size_t)Wp * sizeof(float), noise + r.pa, (size_t)T * sizeof(float),
                                   (size_t)Wp * sizeof(float), (size_t)B * H, cudaMemcpyDeviceToDevice, st));
  else
    VSG_TRY(launch_noise(seeds, nz, B, H, Wp, st, r.pa));
  // z = posterior_encoder(spectrogram(wav), mask, g_src) over [pa, pb), the rows framed from the caller's wav in place
  if (bf) {
    VSG_TRY(spectrogram_tc(P, S, en.in_pad, wav, lengths, mask_p, u, B, Wp, ws, st, r.pa, T));
    VSG_TRY(posterior_core_tc(m.post, u, mask_p, g_src, nz, z, stats, B, Wp, ws, st));
  } else {
    const size_t mark = ws.off;
    VSG_TRY(spectrogram_f32(S, wav, lengths, mask_p, x, B, Wp, ws, st, r.pa, T));
    ws.off = mark;
    VSG_TRY(posterior_forward_f32(m.post, x, mask_p, g_src, nz, z, stats, B, Wp, ws, st));
  }
  // z_p = flow(z, mask, g_src) over [ga, gb), read in place from the posterior's rows
  ws.off = mark0;
  VSG_TRY(run_flow(hot, z + (r.ga - r.pa), mask_p + (r.ga - r.pa), g_src, z_p, B, Wg, 0, precision, ws, st, nullptr,
                   nullptr, nullptr, nullptr, Wp));
  // flow reverse under g_tgt and the decoder: the streaming-synthesis window body on z_p's rows
  ws.off = mark0;
  return zp_window_run(hot, z_p, mask_g, r.ga, Wg, g_tgt, wav_out, wav_ld, z_out, B, T, t0, t1, precision, ws, st);
}

// ---- pack creation --------------------------------------------------------------------------------------------------

const VsgTensor* find_weight(const VsgTensor* w, int n, const std::string& name) {
  for (int i = 0; i < n; ++i)
    if (w[i].name && name == w[i].name) return &w[i];
  return nullptr;
}

int64_t numel(const VsgTensor& t) {
  int64_t n = 1;
  for (int d = 0; d < t.ndim; ++d) n *= t.shape[d];
  return n;
}

int check_config(const VsgModelConfig& c) {
  if (c.ph_dict_size <= 0 || c.pitch_size <= 0 || c.dur_size <= 0)
    return fail(VSG_EINVAL, "bad model config: dictionary sizes %d / %d / %d", c.ph_dict_size, c.pitch_size, c.dur_size);
  if (c.hidden <= 0 || c.filter <= 0 || c.n_heads <= 0 || c.hidden % c.n_heads || c.ffn_kernel_size <= 0 ||
      c.ffn_kernel_size % 2 == 0 || c.window_size < 0 || c.enc_layers <= 0 || c.frame_prior_layers <= 0 ||
      (c.use_pitch_embed && c.pitch_predictor_layers <= 0))
    return fail(VSG_EINVAL, "bad model config (hidden %d filter %d heads %d kernel %d window %d layers %d / %d / %d)", c.hidden,
                c.filter, c.n_heads, c.ffn_kernel_size, c.window_size, c.enc_layers, c.pitch_predictor_layers,
                c.frame_prior_layers);
  if (!c.use_spk_id && !c.use_spk_embed)
    return fail(VSG_EINVAL, "bad model config: VISinger conditions on a speaker (use_spk_id or use_spk_embed)");
  if ((c.use_spk_id && c.num_spk <= 0) || (c.use_spk_embed && c.spk_embed_dim <= 0))
    return fail(VSG_EINVAL, "bad model config: num_spk %d, spk_embed_dim %d", c.num_spk, c.spk_embed_dim);
  if (c.hidden < 4) return fail(VSG_EINVAL, "bad model config: the position table needs hidden >= 4");
  const VsgConfig& h = c.hot;
  if (h.flow_n_flows <= 0 || h.dec_n_ups <= 0 || h.flow_channels != c.hidden || h.dec_initial_channel != c.hidden ||
      h.flow_gin <= 0 || h.flow_gin != h.dec_gin)
    return fail(VSG_EINVAL, "bad model config: the flow and decoder take hidden = %d channels and one speaker condition "
                "(flow channels %d, decoder initial_channel %d, gin %d / %d)", c.hidden, h.flow_channels,
                h.dec_initial_channel, h.flow_gin, h.dec_gin);
  return VSG_OK;
}

// The window-folded DFT basis (spec.cuh, SpecPack), evaluated in double with the phase k * n reduced mod n_fft exactly,
// rounded once to fp32: the FFMA pack [hop][taps][CoutP]; the tcgen05 pack rounds those values to bf16, like every
// other weight, into Cout = 2 * in_pad rows (zero pad pairs) of hopP channels.  A periodic Hann window of win samples,
// zero-padded centrally to n_fft as torch.stft does.
int pack_spec(VsgPack* P, SpecPack& S, int in_pad) {
  const int N = S.n_fft, W = S.win, h = S.hop, K = S.taps, bins = S.bins, lead = (N - W) / 2;
  const int Cout = 2 * bins, CoutP = (Cout + 63) / 64 * 64, CoutT = 2 * in_pad;
  std::vector<float> wf((size_t)h * K * CoutP, 0.f), wt((size_t)CoutT * S.hopP * K, 0.f), bt(CoutT, 0.f);
  const double two_pi = 6.283185307179586476925286766559;
  for (int t = 0; t < K; ++t)
    for (int j = 0; j < h; ++j) {
      const int nr = t * h + j;               // sample inside the window
      if (nr >= W) continue;
      const long long n = lead + nr;          // sample inside the n_fft frame
      const double w = 0.5 - 0.5 * cos(two_pi * nr / W);
      for (int k = 0; k < bins; ++k) {
        const double a = two_pi * (double)((k * n) % N) / N;
        const float re = (float)(w * cos(a)), im = (float)(-w * sin(a));
        wf[((size_t)j * K + t) * CoutP + 2 * k] = re;
        wf[((size_t)j * K + t) * CoutP + 2 * k + 1] = im;
        wt[((size_t)(2 * k) * S.hopP + j) * K + t] = re;
        wt[((size_t)(2 * k + 1) * S.hopP + j) * K + t] = im;
      }
    }
  void* q = nullptr;
  VSG_CUDA_TRY(cudaMalloc(&q, wf.size() * sizeof(float)));
  P->allocs.push_back(q);
  VSG_CUDA_TRY(cudaMemcpy(q, wf.data(), wf.size() * sizeof(float), cudaMemcpyHostToDevice));
  S.f32.w = (float*)q;
  S.f32.bias = nullptr;
  S.f32.Cin = h; S.f32.Cout = Cout; S.f32.CoutP = CoutP; S.f32.ktaps = K;
  return pack_conv_tc(P, wt, bt, CoutT, S.hopP, K, &S.tc);
}

}  // namespace

void model_pack_free(ModelPack* m) {
  vsg_pack_destroy(m->post);
  vsg_pack_destroy(m->text);
  vsg_pack_destroy(m->pitch);
  vsg_pack_destroy(m->prior);
  vsg_pack_destroy(m->hot);
  delete m;
}

}  // namespace vsg

using namespace vsg;

extern "C" int vsg_model_pack_create(const VsgModelConfig* cfg, const VsgTensor* weights, int32_t n_weights,
                                     const char* prefix, int32_t device, VsgPack** out) {
  if (!cfg || !out || (!weights && n_weights > 0) || n_weights < 0) return fail(VSG_EINVAL, "null argument");
  *out = nullptr;
  VSG_TRY(check_config(*cfg));
  const VsgModelConfig& c = *cfg;
  const std::string p = prefix ? prefix : "";
  const int H = c.hidden, gin = c.hot.flow_gin;
  // the token-rate weights, host side: every required entry and its size before anything is built
  struct Want { std::string name; int64_t n; bool need; std::vector<float>* dst; };
  std::vector<float> ph, pt, du, lw, lb, sw, sew, seb, pw, pb, fq;
  std::vector<Want> want = {
      {"text_encoder.ph_emb.weight", (int64_t)c.ph_dict_size * H, true, &ph},
      {"text_encoder.pitch_emb.weight", (int64_t)c.pitch_size * H, true, &pt},
      {"text_encoder.dur_emb.weight", (int64_t)c.dur_size * H, true, &du},
      {"text_encoder.linear.weight", (int64_t)3 * H * H, true, &lw},
      {"text_encoder.linear.bias", H, true, &lb},
      {"spk_id_proj.weight", (int64_t)c.num_spk * gin, c.use_spk_id != 0, &sw},
      {"spk_embed_proj.weight", (int64_t)gin * c.spk_embed_dim, c.use_spk_embed != 0, &sew},
      {"spk_embed_proj.bias", gin, c.use_spk_embed != 0, &seb},
      {"pitch_predictor.linear.weight", (int64_t)2 * H, c.use_pitch_embed != 0, &pw},
      {"pitch_predictor.linear.bias", 2, c.use_pitch_embed != 0, &pb},
      {"embed_positions.freq", H / 2, false, &fq},
  };
  for (Want& w : want) {
    const VsgTensor* t = find_weight(weights, n_weights, p + w.name);
    if (!t) {
      if (w.need) return fail(VSG_EINVAL, "missing weight %s%s", p.c_str(), w.name.c_str());
      continue;
    }
    if (!t->data || t->ndim < 0 || t->ndim > 4 || numel(*t) != w.n)
      return fail(VSG_EINVAL, "weight %s%s is malformed or has the wrong size (expected %lld elements)", p.c_str(),
                  w.name.c_str(), (long long)w.n);
    w.dst->assign(t->data, t->data + w.n);
  }
  int ndev = 0;
  VSG_CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(VSG_EINVAL, "device %d out of range (%d visible)", device, ndev);
  struct Restore { int prev = -1; ~Restore() { if (prev >= 0) cudaSetDevice(prev); } } restore;
  VSG_CUDA_TRY(cudaGetDevice(&restore.prev));
  VSG_CUDA_TRY(cudaSetDevice(device));
  VsgPack* P = new VsgPack();
  memset(&P->cfg, 0, sizeof(P->cfg));
  P->device = device;
  ModelPack* m = new ModelPack();
  P->model = m;
  m->cfg = c;
  m->gin = gin;
  auto upload = [&](const std::vector<float>& h, const float** d) -> int {
    if (h.empty()) return VSG_OK;
    void* q = nullptr;
    VSG_CUDA_TRY(cudaMalloc(&q, h.size() * sizeof(float)));
    P->allocs.push_back(q);
    VSG_CUDA_TRY(cudaMemcpy(q, h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice));
    *d = (const float*)q;
    return VSG_OK;
  };
  auto build = [&]() -> int {
    const VsgRelEncConfig te = {H, c.filter, c.n_heads, c.enc_layers, c.ffn_kernel_size, c.window_size, 0};
    VSG_TRY(vsg_relenc_pack_create(&te, weights, n_weights, (p + "text_encoder.text_encoder.").c_str(), device, &m->text));
    if (c.use_pitch_embed) {
      const VsgRelEncConfig pe = {H, c.filter, c.n_heads, c.pitch_predictor_layers, c.ffn_kernel_size, c.window_size, gin};
      VSG_TRY(vsg_relenc_pack_create(&pe, weights, n_weights, (p + "pitch_predictor.pitch_predictor.").c_str(), device,
                                     &m->pitch));
    }
    const VsgRelEncConfig fp = {H, c.filter, c.n_heads, c.frame_prior_layers, c.ffn_kernel_size, c.window_size, 1};
    VSG_TRY(vsg_frame_prior_pack_create(&fp, weights, n_weights, (p + "frame_prior.").c_str(), device, &m->prior));
    VSG_TRY(vsg_pack_create(&c.hot, weights, n_weights, (p + "flow.").c_str(), (p + "decoder.").c_str(), device, &m->hot));
    std::vector<float> lwt((size_t)3 * H * H);   // [H][3H] -> [3H][H]
    for (int o = 0; o < H; ++o)
      for (int k = 0; k < 3 * H; ++k) lwt[(size_t)k * H + o] = lw[(size_t)o * 3 * H + k];
    VSG_TRY(upload(ph, &m->ph_emb));
    VSG_TRY(upload(pt, &m->pitch_emb));
    VSG_TRY(upload(du, &m->dur_emb));
    VSG_TRY(upload(lwt, &m->lin_wt));
    VSG_TRY(upload(lb, &m->lin_b));
    VSG_TRY(upload(sw, &m->spk_id_w));
    VSG_TRY(upload(sew, &m->spk_embed_w));
    VSG_TRY(upload(seb, &m->spk_embed_b));
    VSG_TRY(upload(pw, &m->pitch_w));
    VSG_TRY(upload(pb, &m->pitch_b));
    VSG_TRY(upload(fq, &m->freq));
    return VSG_OK;
  };
  const int rc = build();
  if (rc != VSG_OK) {
    vsg_pack_destroy(P);
    return rc;
  }
  *out = P;
  return VSG_OK;
}

extern "C" size_t vsg_model_workspace_bytes(const VsgPack* pack, int32_t B, int32_t T_ph, int32_t T, int32_t precision) {
  if (!pack || !pack->model || B < 0 || T_ph < 0 || T < 0 || B > 65535) return 0;
  if (precision != VSG_PRECISION_FP32 && precision != VSG_PRECISION_BF16 && precision != VSG_PRECISION_BF16X3) return 0;
  return model_ws_bytes(pack, B, T_ph, T, precision);
}

extern "C" int vsg_model_forward(const VsgPack* pack, const int64_t* text_tokens, const int64_t* pitch_tokens,
                                 const int64_t* dur_tokens, const int64_t* mel2ph, const int64_t* spk_id,
                                 const float* spk_embed, const float* f0, const float* uv, const float* noise,
                                 const uint64_t* seeds, float* wav, float* f0_pred, float* z_q_out, int32_t B, int32_t T_ph,
                                 int32_t T, int32_t precision, void* workspace, size_t workspace_bytes, void* stream) {
  reset_launch_counts();
  if (!pack || !pack->model) return fail(VSG_EINVAL, "pack is not a model pack (create it with vsg_model_pack_create)");
  const ModelPack& m = *pack->model;
  const VsgModelConfig& c = m.cfg;
  if (B < 0 || T_ph < 0 || T < 0) return fail(VSG_EINVAL, "negative batch (%d) or length (%d, %d)", B, T_ph, T);
  if (B > 65535) return fail(VSG_EUNSUPPORTED, "batch %d exceeds 65535", B);
  if (precision != VSG_PRECISION_FP32 && precision != VSG_PRECISION_BF16 && precision != VSG_PRECISION_BF16X3)
    return fail(VSG_EINVAL, "unknown precision %d", precision);
  if (B == 0 || T == 0) return VSG_OK;
  if (T_ph == 0) return fail(VSG_EINVAL, "T_ph is 0 but T is %d: frames need tokens", T);
  if ((long long)T * vsg_hop_size(m.hot) > 0x7fffffffLL / 4) return fail(VSG_EUNSUPPORTED, "sequence too long (%d frames)", T);
  if (!text_tokens || !pitch_tokens || !dur_tokens || !mel2ph || !wav)
    return fail(VSG_EINVAL, "null pointer: text_tokens, pitch_tokens, dur_tokens, mel2ph and wav are required");
  if (c.use_spk_id != (spk_id != nullptr))
    return fail(VSG_EINVAL, c.use_spk_id ? "spk_id is required (use_spk_id)" : "spk_id given but the model has no use_spk_id");
  if (c.use_spk_embed != (spk_embed != nullptr))
    return fail(VSG_EINVAL, c.use_spk_embed ? "spk_embed is required (use_spk_embed)"
                                            : "spk_embed given but the model has no use_spk_embed");
  if ((f0 == nullptr) != (uv == nullptr)) return fail(VSG_EINVAL, "f0 and uv come together (both or neither)");
  if (!c.use_pitch_embed && (f0 || f0_pred))
    return fail(VSG_EINVAL, "f0 / uv / f0_pred given but the model has no pitch predictor (use_pitch_embed)");
  if (!noise && !seeds) return fail(VSG_EINVAL, "noise and seeds are both NULL: one of them is required");
  if (spk_id)
    for (int b = 0; b < B; ++b)
      if (spk_id[b] < 0 || spk_id[b] >= c.num_spk)
        return fail(VSG_EINVAL, "spk_id[%d] = %lld is outside [0, %d)", b, (long long)spk_id[b], c.num_spk);
  const size_t need = model_ws_bytes(pack, B, T_ph, T, precision);
  if (!workspace || workspace_bytes < need)
    return fail(VSG_ENOMEM, "workspace of %zu bytes is too small: need %zu", workspace ? workspace_bytes : (size_t)0, need);
  DeviceGuard dg(pack->device);
  if (!dg.ok) return fail(VSG_ECUDA, "cannot select device %d", pack->device);
  Workspace ws(workspace, workspace_bytes);
  return model_forward(pack, (const long long*)text_tokens, (const long long*)pitch_tokens, (const long long*)dur_tokens,
                       (const long long*)mel2ph, spk_id, spk_embed, f0, uv, noise, seeds, wav, f0_pred, z_q_out, B, T_ph, T,
                       precision, ws, (cudaStream_t)stream);
}

extern "C" int vsg_normal_noise(const uint64_t* seeds, float* out, int32_t B, int32_t C, int32_t T, void* stream) {
  reset_launch_counts();
  if (B < 0 || C < 0 || T < 0) return fail(VSG_EINVAL, "negative dimension");
  if ((long long)B * C * T == 0) return VSG_OK;
  if (!seeds || !out) return fail(VSG_EINVAL, "null pointer");
  return launch_noise(seeds, out, B, C, T, (cudaStream_t)stream);
}

extern "C" int vsg_debug_position_table(const float* freq, int32_t rows, int32_t dim, float* out, void* stream) {
  reset_launch_counts();
  if (rows < 0 || dim < 4) return fail(VSG_EINVAL, "bad table shape (%d rows, dim %d; dim >= 4)", rows, dim);
  if (rows == 0) return VSG_OK;
  if (!out) return fail(VSG_EINVAL, "null pointer");
  return launch_prep(nullptr, nullptr, 0, freq, out, rows, dim, (cudaStream_t)stream);
}

extern "C" int vsg_convert_pack_create(const VsgModelConfig* cfg, const VsgTensor* weights, int32_t n_weights,
                                       const char* prefix, int32_t win_length, int32_t device, VsgPack** out) {
  if (!cfg || !out || (!weights && n_weights > 0) || n_weights < 0) return fail(VSG_EINVAL, "null argument");
  *out = nullptr;
  VSG_TRY(check_config(*cfg));
  const VsgModelConfig& c = *cfg;
  const std::string p = prefix ? prefix : "";
  const std::string pe = p + "posterior_encoder.";
  // PosteriorEncoder(num_linear_bins, hidden, hidden, kernel_size, 1, n_layers, gin) (models/visinger.py:59-60): the bins,
  // kernel and layer count come from the weights, the dilation rate is VISinger's 1
  const VsgTensor* pre = find_weight(weights, n_weights, pe + "pre.weight");
  if (!pre) return fail(VSG_EINVAL, "missing weight %spre.weight", pe.c_str());
  if (!pre->data || pre->ndim < 2 || pre->ndim > 3 || pre->shape[0] != c.hidden || pre->shape[1] < 2 ||
      (pre->ndim == 3 && pre->shape[2] != 1))
    return fail(VSG_EINVAL, "weight %spre.weight must be [hidden = %d, bins >= 2, 1]", pe.c_str(), c.hidden);
  const VsgTensor* proj = find_weight(weights, n_weights, pe + "proj.weight");
  if (!proj) return fail(VSG_EINVAL, "missing weight %sproj.weight", pe.c_str());
  if (proj->ndim < 2 || proj->shape[0] != 2 * c.hidden)
    return fail(VSG_EINVAL, "weight %sproj.weight must have 2 * hidden = %d output channels (the flow's)", pe.c_str(),
                2 * c.hidden);
  auto in_layer = [&](int i) {
    const std::string k = pe + "enc.in_layers." + std::to_string(i);
    const VsgTensor* t = find_weight(weights, n_weights, k + ".weight");
    return t ? t : find_weight(weights, n_weights, k + ".weight_v");
  };
  int n_layers = 0;
  while (in_layer(n_layers)) ++n_layers;
  if (n_layers == 0) return fail(VSG_EINVAL, "missing weight %senc.in_layers.0.weight (or .weight_v)", pe.c_str());
  const VsgTensor* l0 = in_layer(0);
  if (l0->ndim != 3) return fail(VSG_EINVAL, "weight %senc.in_layers.0 must be [2 * hidden, hidden, kernel]", pe.c_str());
  const int bins = (int)pre->shape[1], n_fft = 2 * (bins - 1);
  int hop = 1;
  for (int i = 0; i < c.hot.dec_n_ups && i < VSG_MAX_UPS; ++i) hop *= c.hot.dec_upsample_rates[i];
  if (win_length <= 0 || win_length > n_fft)
    return fail(VSG_EINVAL, "win_length %d is outside [1, n_fft = %d] (n_fft = 2 * (bins - 1), bins = %d)", win_length, n_fft,
                bins);
  if (n_fft < hop) return fail(VSG_EINVAL, "n_fft %d is below the decoder's hop %d: frames would skip samples", n_fft, hop);

  VsgPack* P = nullptr;
  VSG_TRY(vsg_model_pack_create(cfg, weights, n_weights, prefix, device, &P));
  struct Restore { int prev = -1; ~Restore() { if (prev >= 0) cudaSetDevice(prev); } } restore;
  auto build = [&]() -> int {
    ModelPack& m = *P->model;
    const VsgEncConfig ec = {bins, c.hidden, c.hidden, (int32_t)l0->shape[2], 1, n_layers, m.gin};
    VSG_TRY(vsg_enc_pack_create(&ec, weights, n_weights, pe.c_str(), device, &m.post));
    SpecPack& S = m.spec;
    S.n_fft = n_fft; S.win = win_length; S.hop = hop; S.bins = bins;
    S.taps = (win_length + hop - 1) / hop;
    S.off = (n_fft - win_length) / 2 - (n_fft - hop) / 2;
    S.hopP = (hop + 63) / 64 * 64;
    VSG_CUDA_TRY(cudaGetDevice(&restore.prev));
    VSG_CUDA_TRY(cudaSetDevice(device));
    return pack_spec(P, S, m.post->enc.in_pad);
  };
  const int rc = build();
  if (rc != VSG_OK) {
    vsg_pack_destroy(P);
    return rc;
  }
  *out = P;
  return VSG_OK;
}

extern "C" size_t vsg_convert_workspace_bytes(const VsgPack* pack, int32_t B, int32_t T, int32_t precision) {
  if (!pack || !pack->model || !pack->model->post || B < 0 || T < 0 || B > 65535) return 0;
  if (precision != VSG_PRECISION_FP32 && precision != VSG_PRECISION_BF16 && precision != VSG_PRECISION_BF16X3) return 0;
  return convert_ws_bytes(pack, B, T, precision);
}

namespace {

int check_convert(const VsgPack* pack, int B, int T, int precision) {
  if (!pack || !pack->model || !pack->model->post)
    return fail(VSG_EINVAL, "pack has no posterior encoder or spectrogram (create it with vsg_convert_pack_create)");
  if (B < 0 || T < 0) return fail(VSG_EINVAL, "negative batch (%d) or length (%d)", B, T);
  if (B > 65535) return fail(VSG_EUNSUPPORTED, "batch %d exceeds 65535", B);
  if (precision != VSG_PRECISION_FP32 && precision != VSG_PRECISION_BF16 && precision != VSG_PRECISION_BF16X3)
    return fail(VSG_EINVAL, "unknown precision %d", precision);
  if ((long long)T * pack->model->spec.hop > 0x7fffffffLL / 4) return fail(VSG_EUNSUPPORTED, "sequence too long (%d frames)", T);
  return VSG_OK;
}

// the speaker and noise arguments of vsg_model_convert / vsg_model_convert_window (host ids range-checked)
int check_convert_inputs(const VsgModelConfig& c, int B, const int64_t* src_spk_id, const float* src_spk_embed,
                         const int64_t* tgt_spk_id, const float* tgt_spk_embed, const float* noise, const uint64_t* seeds) {
  if (c.use_spk_id != (src_spk_id != nullptr) || c.use_spk_id != (tgt_spk_id != nullptr))
    return fail(VSG_EINVAL, c.use_spk_id ? "src_spk_id and tgt_spk_id are required (use_spk_id)"
                                         : "speaker ids given but the model has no use_spk_id");
  if (c.use_spk_embed != (src_spk_embed != nullptr) || c.use_spk_embed != (tgt_spk_embed != nullptr))
    return fail(VSG_EINVAL, c.use_spk_embed ? "src_spk_embed and tgt_spk_embed are required (use_spk_embed)"
                                            : "speaker embeddings given but the model has no use_spk_embed");
  if (!noise && !seeds) return fail(VSG_EINVAL, "noise and seeds are both NULL: one of them is required");
  for (const int64_t* ids : {src_spk_id, tgt_spk_id})
    if (ids)
      for (int b = 0; b < B; ++b)
        if (ids[b] < 0 || ids[b] >= c.num_spk)
          return fail(VSG_EINVAL, "%s_spk_id[%d] = %lld is outside [0, %d)", ids == src_spk_id ? "src" : "tgt", b,
                      (long long)ids[b], c.num_spk);
  return VSG_OK;
}

// a window [t0, t1) of a (B, T) batch: where the window call's arguments differ from the one-pass call's
int check_convert_window(const VsgPack* pack, int B, int T, int t0, int t1, int precision) {
  VSG_TRY(check_convert(pack, B, T, precision));
  if (t0 < 0 || t1 > T || t0 >= t1) return fail(VSG_EINVAL, "window [%d, %d) is not a non-empty part of [0, %d)", t0, t1, T);
  WinRange r;   // (a kernel the whole batch chooses with no window form: VSG_EUNSUPPORTED)
  if (B > 0) VSG_TRY(window_ranges(pack->model->hot, B, T, t0, t1, precision, true, &r, post_context(*pack->model)));
  return VSG_OK;
}

}  // namespace

extern "C" int vsg_spectrogram(const VsgPack* pack, const float* wav, const int32_t* lengths, float* spec, int32_t B,
                               int32_t T, int32_t precision, void* workspace, size_t workspace_bytes, void* stream) {
  reset_launch_counts();
  VSG_TRY(check_convert(pack, B, T, precision));
  if (B == 0 || T == 0) return VSG_OK;
  if (!wav || !lengths || !spec) return fail(VSG_EINVAL, "null pointer: wav, lengths and spec are required");
  const size_t need = spectrogram_ws_bytes(pack, B, T, precision);
  if (!workspace || workspace_bytes < need)
    return fail(VSG_ENOMEM, "workspace of %zu bytes is too small: need %zu", workspace ? workspace_bytes : (size_t)0, need);
  DeviceGuard dg(pack->device);
  if (!dg.ok) return fail(VSG_ECUDA, "cannot select device %d", pack->device);
  const ModelPack& m = *pack->model;
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(workspace, workspace_bytes);
  float* mask = ws.take<float>((size_t)B * T);
  if (!convert_bf16(precision)) {
    if (ws.overflow) return fail(VSG_ENOMEM, "spectrogram workspace too small");
    VSG_TRY(lengths_mask(lengths, mask, B, T, st));
    return spectrogram_f32(m.spec, wav, lengths, mask, spec, B, T, ws, st);
  }
  const int in_pad = m.post->enc.in_pad;
  __nv_bfloat16* u = ws.take<__nv_bfloat16>((size_t)B * T * in_pad);
  if (ws.overflow) return fail(VSG_ENOMEM, "spectrogram workspace too small");
  VSG_TRY(lengths_mask(lengths, mask, B, T, st));
  VSG_TRY(spectrogram_tc(pack, m.spec, in_pad, wav, lengths, mask, u, B, T, ws, st));
  return widen_bf16(u, spec, B, m.spec.bins, in_pad, T, st);
}

extern "C" int vsg_model_convert(const VsgPack* pack, const float* wav, const float* spec, const int32_t* lengths,
                                 const int64_t* src_spk_id, const float* src_spk_embed, const int64_t* tgt_spk_id,
                                 const float* tgt_spk_embed, const float* noise, const uint64_t* seeds, float* wav_out,
                                 float* spec_out, float* z_out, int32_t B, int32_t T, int32_t precision, void* workspace,
                                 size_t workspace_bytes, void* stream) {
  reset_launch_counts();
  VSG_TRY(check_convert(pack, B, T, precision));
  const VsgModelConfig& c = pack->model->cfg;
  if (B == 0 || T == 0) return VSG_OK;
  if ((wav == nullptr) == (spec == nullptr)) return fail(VSG_EINVAL, "give exactly one of wav and spec");
  if (spec && spec_out) return fail(VSG_EINVAL, "spec_out receives the spectrogram of wav: it must be NULL when spec is given");
  if (!lengths || !wav_out) return fail(VSG_EINVAL, "null pointer: lengths and wav_out are required");
  VSG_TRY(check_convert_inputs(c, B, src_spk_id, src_spk_embed, tgt_spk_id, tgt_spk_embed, noise, seeds));
  const size_t need = convert_ws_bytes(pack, B, T, precision);
  if (!workspace || workspace_bytes < need)
    return fail(VSG_ENOMEM, "workspace of %zu bytes is too small: need %zu", workspace ? workspace_bytes : (size_t)0, need);
  DeviceGuard dg(pack->device);
  if (!dg.ok) return fail(VSG_ECUDA, "cannot select device %d", pack->device);
  Workspace ws(workspace, workspace_bytes);
  return model_convert(pack, wav, spec, lengths, src_spk_id, src_spk_embed, tgt_spk_id, tgt_spk_embed, noise, seeds,
                       wav_out, spec_out, z_out, B, T, precision, ws, (cudaStream_t)stream);
}

extern "C" int vsg_convert_window_context(const VsgPack* pack, int32_t* post_frames, int32_t* flow_frames,
                                          int32_t* dec_frames) {
  if (!pack || !pack->model || !pack->model->post)
    return fail(VSG_EINVAL, "pack has no posterior encoder or spectrogram (create it with vsg_convert_pack_create)");
  if (!post_frames || !flow_frames || !dec_frames) return fail(VSG_EINVAL, "null pointer");
  *post_frames = post_context(*pack->model);
  *flow_frames = flow_context(pack->model->hot);
  *dec_frames = dec_context(pack->model->hot);
  return VSG_OK;
}

extern "C" int vsg_convert_window_input(const VsgPack* pack, int32_t B, int32_t T, int32_t t0, int32_t t1,
                                        int32_t precision, int64_t* s0, int64_t* s1) {
  VSG_TRY(check_convert_window(pack, B, T, t0, t1, precision));
  if (!s0 || !s1) return fail(VSG_EINVAL, "null pointer");
  WinRange r;
  VSG_TRY(window_ranges(pack->model->hot, std::max(B, 1), T, t0, t1, precision, true, &r, post_context(*pack->model)));
  // spectrogram frames [pa, pb) read rows pa .. pb + taps - 2, row q holding samples [q * hop + off, (q + 1) * hop + off);
  // the mask of frames up to pb - 1 is set by samples below pb * hop
  const SpecPack& S = pack->model->spec;
  const long long hop = S.hop;
  *s0 = std::max(0LL, r.pa * hop + S.off);
  *s1 = std::min((long long)T * hop, std::max(r.pb * hop, (r.pb + S.taps - 1) * hop + S.off));
  return VSG_OK;
}

extern "C" size_t vsg_convert_window_workspace_bytes(const VsgPack* pack, int32_t B, int32_t T, int32_t max_frames,
                                                     int32_t precision) {
  if (!pack || !pack->model || !pack->model->post || B < 0 || T < 0 || B > 65535) return 0;
  if (precision != VSG_PRECISION_FP32 && precision != VSG_PRECISION_BF16 && precision != VSG_PRECISION_BF16X3) return 0;
  return convert_window_ws_bytes(pack, B, T, max_frames, precision);
}

extern "C" int vsg_model_convert_window(const VsgPack* pack, const float* wav, const int32_t* lengths,
                                        const int64_t* src_spk_id, const float* src_spk_embed, const int64_t* tgt_spk_id,
                                        const float* tgt_spk_embed, const float* noise, const uint64_t* seeds,
                                        float* wav_out, int64_t wav_ld, float* z_out, int32_t B, int32_t T, int32_t t0,
                                        int32_t t1, int32_t precision, void* workspace, size_t workspace_bytes,
                                        void* stream) {
  reset_launch_counts();
  VSG_TRY(check_convert_window(pack, B, T, t0, t1, precision));
  if (B == 0) return VSG_OK;
  if (!wav || !lengths || !wav_out) return fail(VSG_EINVAL, "null pointer: wav, lengths and wav_out are required");
  const int hop = pack->model->spec.hop;
  if (wav_ld < (int64_t)(t1 - t0) * hop)
    return fail(VSG_EINVAL, "wav_ld %lld is shorter than the window's %lld samples", (long long)wav_ld,
                (long long)(t1 - t0) * hop);
  VSG_TRY(check_convert_inputs(pack->model->cfg, B, src_spk_id, src_spk_embed, tgt_spk_id, tgt_spk_embed, noise, seeds));
  const size_t need = convert_window_ws_bytes(pack, B, T, t1 - t0, precision);
  if (!workspace || workspace_bytes < need)
    return fail(VSG_ENOMEM, "window workspace of %zu bytes is too small: need %zu", workspace ? workspace_bytes : (size_t)0,
                need);
  DeviceGuard dg(pack->device);
  if (!dg.ok) return fail(VSG_ECUDA, "cannot select device %d", pack->device);
  Workspace ws(workspace, workspace_bytes);
  return model_convert_window(pack, wav, lengths, src_spk_id, src_spk_embed, tgt_spk_id, tgt_spk_embed, noise, seeds,
                              wav_out, wav_ld, z_out, B, T, t0, t1, precision, ws, (cudaStream_t)stream);
}
