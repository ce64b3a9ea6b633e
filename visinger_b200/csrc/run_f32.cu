// fp32 parity-mode drivers: sequence the fused FFMA kernels of kernels_f32.cuh over one batch.
#include "vsg_common.cuh"
#include "kernels_f32.cuh"
#include "relenc_f32.cuh"
#include "run.cuh"
#include "pack_tc.cuh"
#include "spec.cuh"

namespace vsg {

// The tile configuration of conv_f32_kernel for Cout output channels (8 warps: WARPS_CO x WARPS_Q, each 8 channels x 256
// rows) and its dynamic shared memory for k taps at dilation dil: a [8][Q_TILE + halo] input window and the [8][k][CO_TILE]
// weights of one 8-channel chunk.  VSG_EUNSUPPORTED above 200 KB.  The launcher and vsg_debug_conv_f32_plan both use it.
int conv_f32_plan(int Cout, int ktaps, int dil, int* warps_co, int* warps_q, size_t* smem) {
  if (ktaps < 1) return fail(VSG_EUNSUPPORTED, "convolution with no taps");
  const int wc = Cout <= 16 ? 2 : Cout <= 32 ? 4 : 8, wq = 8 / wc;
  const size_t sm = (size_t)F32_CI_CHUNK * ((256 * wq + (size_t)(ktaps - 1) * dil) + (size_t)ktaps * 8 * wc) * sizeof(float);
  if (sm > 200 * 1024) return fail(VSG_EUNSUPPORTED, "conv window too large for shared memory (%zu B)", sm);
  *warps_co = wc; *warps_q = wq; *smem = sm;
  return VSG_OK;
}

namespace {

template <int WC, int WQ, bool MAG>
int launch_conv_f32_tile(const ConvF32& p, int B, size_t sm, cudaStream_t st) {
  if (sm > 48 * 1024)
    VSG_CUDA_TRY(cudaFuncSetAttribute(conv_f32_kernel<WC, WQ, MAG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  dim3 grid((p.Lq + 256 * WQ - 1) / (256 * WQ), (p.Cout + 8 * WC - 1) / (8 * WC), B);
  conv_f32_kernel<WC, WQ, MAG><<<grid, 256, sm, st>>>(p);
  VSG_LAUNCH_CHECK("conv_f32_kernel");
  return VSG_OK;
}

// tile_out (optional): the (WARPS_CO, WARPS_Q) configuration launched.
template <bool MAG = false>
int launch_conv_f32(const ConvF32& p, int B, cudaStream_t st, int* tile_out = nullptr) {
  if (p.ktaps < 1) return fail(VSG_EUNSUPPORTED, "convolution with no taps");
  if (p.Lq <= 0) return VSG_OK;
  int wc = 0, wq = 0;
  size_t sm = 0;
  VSG_TRY(conv_f32_plan(p.Cout, p.ktaps, p.dil, &wc, &wq, &sm));
  if (tile_out) { tile_out[0] = wc; tile_out[1] = wq; }
  if (wc == 2) return launch_conv_f32_tile<2, 4, MAG>(p, B, sm, st);
  if (wc == 4) return launch_conv_f32_tile<4, 2, MAG>(p, B, sm, st);
  return launch_conv_f32_tile<8, 1, MAG>(p, B, sm, st);
}

ConvF32 base_conv(const ConvW32& w, const float* x, long long x_bs, int x_cs, int Lin, int in_off0, int dil) {
  ConvF32 p;
  memset(&p, 0, sizeof(p));
  p.x = x; p.x_bs = x_bs; p.x_cs = x_cs; p.Cin = w.Cin; p.Lin = Lin;
  p.in_off0 = in_off0; p.dil = dil; p.ktaps = w.ktaps;
  p.slope = 0.1f;   // LRELU_SLOPE, modules/visinger/decoder.py:10
  p.w = w.w; p.CoutP = w.CoutP; p.bias = w.bias; p.Cout = w.Cout;
  p.Lq = Lin; p.out_stride = 1; p.out_phase = 0; p.Lout = Lin;
  p.epi = EPI_LINEAR; p.acc_mode = ACC_SET; p.acc_div = 1.f;
  return p;
}

}  // namespace

int launch_cond(const float* W, const float* bias, const float* g, float* out, int O, int I, int B, cudaStream_t st) {
  const long long warps = (long long)O * B;
  const int threads = 256;
  const int blocks = (int)((warps * 32 + threads - 1) / threads);
  cond_gemv_kernel<<<blocks, threads, 0, st>>>(W, bias, g, out, O, I, B);
  VSG_LAUNCH_CHECK("cond_gemv_kernel");
  return VSG_OK;
}

size_t flow_ws_bytes_f32(const VsgPack* P, int B, int T) {
  const VsgConfig& c = P->cfg;
  size_t n = 0;
  n += align256((size_t)B * c.flow_n_flows * 2 * c.flow_hidden * c.flow_n_layers * sizeof(float));  // cond
  n += 3 * align256((size_t)B * c.flow_hidden * T * sizeof(float));                                  // h, acts, out
  return n;
}

// ResidualCouplingBlock.forward, modules/visinger/flow.py:33-40, with the Flips folded away.
int flow_forward_f32(const VsgPack* P, const float* x, const float* mask, const float* g, float* y, int B, int T,
                     int reverse, Workspace& ws, cudaStream_t st, int x_ld) {
  const VsgConfig& c = P->cfg;
  const int C = c.flow_channels, H = c.flow_hidden, NL = c.flow_n_layers, NF = c.flow_n_flows, half = C / 2;
  const int condO = 2 * H * NL;
  const int ld = x_ld > 0 ? x_ld : T;
  float* cond = ws.take<float>((size_t)B * NF * condO);
  float* h = ws.take<float>((size_t)B * H * T);
  float* acts = ws.take<float>((size_t)B * H * T);
  float* out = ws.take<float>((size_t)B * H * T);
  if (ws.overflow) return fail(VSG_ENOMEM, "flow workspace too small: need %zu bytes", ws.off);
  // Each channel half is read from x until a coupling first writes it into y (its epilogue reads the old x1 from x), so
  // the input is never copied -- nor gathered, when x is a window of a longer batch.  (y may alias x.)
  const float* src[2] = {x, x + (long long)half * ld};
  long long src_bs[2] = {(long long)C * ld, (long long)C * ld};
  int src_cs[2] = {ld, ld};
  bool in_y[2] = {false, false};
  if (c.flow_gin > 0) {
    if (!g) return fail(VSG_EINVAL, "flow was built with gin_channels=%d but g is NULL", c.flow_gin);
    for (int f = 0; f < NF; ++f)
      VSG_TRY(launch_cond(P->flow_layers[f].cond_w, P->flow_layers[f].cond_b, g, cond + (size_t)f * condO * B, condO,
                          c.flow_gin, B, st));
  }
  const long long CT = (long long)C * T, HT = (long long)H * T;
  for (int step = 0; step < NF; ++step) {
    const int f = reverse ? NF - 1 - step : step;
    const int flipped = reverse ? (NF - f) & 1 : f & 1;   // parity of Flips applied so far
    const FlowLayer& fl = P->flow_layers[f];
    const int h0 = flipped ? 1 : 0, h1 = 1 - h0;                  // conditioning half (never modified here), updated half
    float* x1 = y + (long long)h1 * half * T;
    // h = pre(x0) * mask                                           flow.py:68
    {
      ConvF32 p = base_conv(fl.pre[flipped], src[h0], src_bs[h0], src_cs[h0], T, 0, 1);
      p.y = h; p.y_bs = HT; p.y_cs = T; p.mask = mask; p.mask_bs = ld;
      VSG_TRY(launch_conv_f32(p, B, st));
    }
    // WaveNet                                                       encoder.py:174-195
    int dil = 1;
    for (int i = 0; i < NL; ++i) {
      const int K = c.flow_kernel_size;
      const int pad = (K * dil - dil) / 2;
      {
        ConvF32 p = base_conv(fl.in_layers[i], h, HT, T, T, -pad, dil);
        p.epi = EPI_GATE;
        if (c.flow_gin > 0) { p.bcond = cond + (size_t)f * condO * B + (size_t)i * 2 * H; p.bcond_bs = condO; }
        p.y = acts; p.y_bs = HT; p.y_cs = T;
        VSG_TRY(launch_conv_f32(p, B, st));
      }
      {
        ConvF32 p = base_conv(fl.res_skip[i], acts, HT, T, T, 0, 1);
        p.epi = EPI_RES_SKIP;
        const bool last = (i == NL - 1);
        p.rs_split = last ? 0 : H;
        p.y = h; p.y_bs = HT; p.y_cs = T;
        p.y2 = out; p.y2_bs = HT; p.y2_cs = T;
        p.y2_first = (i == 0); p.y2_mask = last;
        p.mask = mask; p.mask_bs = ld;
        VSG_TRY(launch_conv_f32(p, B, st));
      }
      dil *= c.flow_dilation_rate;
    }
    // m = post(h) * mask ; x1 = (x1 - m) * mask | m + x1 * mask     flow.py:70,78,83
    {
      ConvF32 p = base_conv(fl.post[flipped], out, HT, T, T, 0, 1);
      p.epi = EPI_COUPLE; p.couple_sign = reverse ? -1 : 1;
      p.y = x1; p.y_bs = CT; p.y_cs = T; p.mask = mask; p.mask_bs = ld;
      if (!in_y[h1]) { p.res = src[h1]; p.res_bs = src_bs[h1]; p.res_cs = src_cs[h1]; }
      VSG_TRY(launch_conv_f32(p, B, st));
    }
    src[h1] = x1; src_bs[h1] = CT; src_cs[h1] = T; in_y[h1] = true;
  }
  for (int hh = 0; hh < 2; ++hh)   // a half no coupling wrote (one flow only) is copied
    if (!in_y[hh] && src[hh] != y + (long long)hh * half * T)
      for (int b = 0; b < B; ++b)
        VSG_CUDA_TRY(cudaMemcpy2DAsync(y + ((long long)b * C + hh * half) * T, (size_t)T * sizeof(float),
                                       src[hh] + (long long)b * C * ld, (size_t)ld * sizeof(float), (size_t)T * sizeof(float),
                                       half, cudaMemcpyDeviceToDevice, st));
  if (NF & 1) {   // an odd number of Flips does not cancel
    const long long n = (long long)B * half * T;
    flip_channels_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(y, C, T, n);
    VSG_LAUNCH_CHECK("flip_channels_kernel");
  }
  return VSG_OK;
}

size_t posterior_ws_bytes_f32(const VsgPack* P, int B, int T) {
  const EncPack& e = P->enc;
  return align256((size_t)B * 2 * e.hidden * e.n_layers * sizeof(float)) + 3 * align256((size_t)B * e.hidden * T * sizeof(float));
}

// PosteriorEncoder.forward, modules/visinger/encoder.py:92-98.
int posterior_forward_f32(const VsgPack* P, const float* x, const float* mask, const float* g, const float* noise,
                          float* z, float* stats, int B, int T, Workspace& ws, cudaStream_t st) {
  const EncPack& e = P->enc;
  const int H = e.hidden, NL = e.n_layers, K = e.kernel, Cin = e.in_channels, Co = e.out_channels;
  const int condO = 2 * H * NL;
  float* cond = ws.take<float>((size_t)B * condO);
  float* h = ws.take<float>((size_t)B * H * T);
  float* acts = ws.take<float>((size_t)B * H * T);
  float* out = ws.take<float>((size_t)B * H * T);
  if (ws.overflow) return fail(VSG_ENOMEM, "posterior workspace too small: need %zu bytes", ws.off);
  if (e.gin > 0) {
    if (!g) return fail(VSG_EINVAL, "posterior encoder was built with gin_channels=%d but g is NULL", e.gin);
    VSG_TRY(launch_cond(e.wn.cond_w, e.wn.cond_b, g, cond, condO, e.gin, B, st));
  }
  const long long HT = (long long)H * T;
  {  // h = pre(x) * mask                                            encoder.py:93
    ConvF32 p = base_conv(e.pre, x, (long long)Cin * T, T, T, 0, 1);
    p.y = h; p.y_bs = HT; p.y_cs = T; p.mask = mask; p.mask_bs = T;
    VSG_TRY(launch_conv_f32(p, B, st));
  }
  int dil = 1;
  for (int i = 0; i < NL; ++i) {   // WaveNet                        encoder.py:174-195
    const int pad = (K * dil - dil) / 2;
    {
      ConvF32 p = base_conv(e.wn.in_layers[i], h, HT, T, T, -pad, dil);
      p.epi = EPI_GATE;
      if (e.gin > 0) { p.bcond = cond + (size_t)i * 2 * H; p.bcond_bs = condO; }
      p.y = acts; p.y_bs = HT; p.y_cs = T;
      VSG_TRY(launch_conv_f32(p, B, st));
    }
    {
      ConvF32 p = base_conv(e.wn.res_skip[i], acts, HT, T, T, 0, 1);
      p.epi = EPI_RES_SKIP;
      const bool last = (i == NL - 1);
      p.rs_split = last ? 0 : H;
      p.y = h; p.y_bs = HT; p.y_cs = T;
      p.y2 = out; p.y2_bs = HT; p.y2_cs = T;
      p.y2_first = (i == 0); p.y2_mask = last;
      p.mask = mask; p.mask_bs = T;
      VSG_TRY(launch_conv_f32(p, B, st));
    }
    dil *= e.dil_rate;
  }
  {  // stats = proj(h) * mask                                        encoder.py:95
    ConvF32 p = base_conv(e.proj, out, HT, T, T, 0, 1);
    p.y = stats; p.y_bs = (long long)2 * Co * T; p.y_cs = T; p.mask = mask; p.mask_bs = T;
    VSG_TRY(launch_conv_f32(p, B, st));
  }
  const long long n = (long long)B * Co * T;   // z = (mu + noise * exp(logs)) * mask   encoder.py:96-97
  posterior_sample_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(stats, noise, mask, z, Co, T, n);
  VSG_LAUNCH_CHECK("posterior_sample_kernel");
  return VSG_OK;
}

int lengths_mask(const int32_t* lengths, float* mask, int B, int T, cudaStream_t st, int t0, int T_len) {
  const long long n = (long long)B * T;
  lengths_mask_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(lengths, mask, T, t0, T_len ? T_len : T, n);
  VSG_LAUNCH_CHECK("lengths_mask_kernel");
  return VSG_OK;
}

// framed rows of the spectrogram: [B, R, hopP] bf16 (tcgen05) or [B, hop, R] fp32 (FFMA), R = T + taps - 1
size_t spec_frames_bytes(const SpecPack& S, int B, int T, bool tc) {
  const size_t R = (size_t)T + S.taps - 1;
  return align256((size_t)B * R * (tc ? S.hopP * 2 : S.hop * 4));
}

// spec [B, bins, T] = |STFT| * mask: the framed rows, then Conv1d(hop -> 2 bins, taps) with the magnitude epilogue.
int spectrogram_f32(const SpecPack& S, const float* wav, const int32_t* lengths, const float* mask, float* spec, int B,
                    int T, Workspace& ws, cudaStream_t st, int t0, int T_len) {
  const int R = T + S.taps - 1;
  if (!T_len) T_len = T;
  float* rows = ws.take<float>((size_t)B * S.hop * R);
  if (ws.overflow) return fail(VSG_ENOMEM, "spectrogram workspace too small: need %zu bytes", ws.off);
  const long long n = (long long)B * S.hop * R;
  spec_frames_kernel<false><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(wav, lengths, rows, T_len, R, S.hop, S.hop, S.off,
                                                                           S.taps, n, t0, (long long)T_len * S.hop);
  VSG_LAUNCH_CHECK("spec_frames_kernel");
  ConvF32 p = base_conv(S.f32, rows, (long long)S.hop * R, R, R, 0, 1);
  p.Lq = T; p.Lout = T;
  p.y = spec; p.y_bs = (long long)S.bins * T; p.y_cs = T; p.mask = mask; p.mask_bs = T;
  return launch_conv_f32<true>(p, B, st);
}

int conv_f32_plain(const ConvW32& w, const float* x, int B, int T, float* y, cudaStream_t st) {
  ConvF32 p = base_conv(w, x, (long long)w.Cin * T, T, T, -(w.ktaps / 2), 1);
  p.y = y; p.y_bs = (long long)w.Cout * T; p.y_cs = T;
  return launch_conv_f32(p, B, st);
}

size_t relenc_ws_bytes_f32(const VsgPack* P, int B, int T, int g_t) {
  const RelEncPack& e = P->relenc;
  size_t n = align256((size_t)B * 3 * e.hidden * T * sizeof(float)) + align256((size_t)B * e.hidden * T * sizeof(float)) +
             align256((size_t)B * e.filter * T * sizeof(float));
  n += align256((size_t)B * e.hidden * (g_t ? T : 1) * sizeof(float));
  return n;
}

namespace {
template <int DK>
int launch_attention_f32(const float* qkv, const float* mask, const float* ek, const float* ev, float* o, int B, int n_heads,
                         int T, int w, cudaStream_t st) {
  const size_t sm = relenc_attention_f32_smem(DK, w);
  if (sm > 200 * 1024) return fail(VSG_EUNSUPPORTED, "attention tile does not fit shared memory (%zu B)", sm);
  VSG_CUDA_TRY(cudaFuncSetAttribute(relenc_attention_f32_kernel<DK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  dim3 grid((T + kAttTile - 1) / kAttTile, n_heads, B);
  relenc_attention_f32_kernel<DK><<<grid, 256, sm, st>>>(qkv, mask, ek, ev, o, n_heads, T, w);
  VSG_LAUNCH_CHECK("relenc_attention_f32_kernel");
  return VSG_OK;
}

int attention_f32(int dk, const float* qkv, const float* mask, const float* ek, const float* ev, float* o, int B, int n_heads,
                  int T, int w, cudaStream_t st) {
  switch (dk) {
    case 16: return launch_attention_f32<16>(qkv, mask, ek, ev, o, B, n_heads, T, w, st);
    case 32: return launch_attention_f32<32>(qkv, mask, ek, ev, o, B, n_heads, T, w, st);
    case 48: return launch_attention_f32<48>(qkv, mask, ek, ev, o, B, n_heads, T, w, st);
    case 64: return launch_attention_f32<64>(qkv, mask, ek, ev, o, B, n_heads, T, w, st);
    case 96: return launch_attention_f32<96>(qkv, mask, ek, ev, o, B, n_heads, T, w, st);
    case 128: return launch_attention_f32<128>(qkv, mask, ek, ev, o, B, n_heads, T, w, st);
    default: return fail(VSG_EUNSUPPORTED, "attention head width %d (supported: 16, 32, 48, 64, 96, 128)", dk);
  }
}
}  // namespace

// RelativeEncoder.forward, modules/rel_transformer.py:286-320 (post-LN; dropout is the identity in eval mode).
// g: NULL, [B, gin] (g_t == 0: one condition vector per utterance, e.g. the speaker embedding) or [B, gin, T] (g_t != 0).
int relenc_forward_f32(const VsgPack* P, const float* x, const float* mask, const float* g, int g_t, float* y, int B, int T,
                       Workspace& ws, cudaStream_t st) {
  const RelEncPack& e = P->relenc;
  const int H = e.hidden, F = e.filter, NL = e.n_layers, K = e.kernel, dk = H / e.n_heads;
  float* qkv = ws.take<float>((size_t)B * 3 * H * T);
  float* o = ws.take<float>((size_t)B * H * T);
  float* f = ws.take<float>((size_t)B * F * T);
  float* gp = ws.take<float>((size_t)B * H * (g_t ? T : 1));
  if (ws.overflow) return fail(VSG_ENOMEM, "encoder workspace too small: need %zu bytes", ws.off);
  const long long HT = (long long)H * T, n = (long long)B * H * T;
  if (g && e.gin <= 0) return fail(VSG_EINVAL, "this encoder has no pre_net (gin_channels is None) but g was given");
  const float* gadd = nullptr;
  if (g) {   // g = pre_net(g)                                        :289-290
    if (g_t) {
      ConvF32 p = base_conv(e.pre_net, g, (long long)e.gin * T, T, T, 0, 1);
      p.y = gp; p.y_bs = HT; p.y_cs = T;
      VSG_TRY(launch_conv_f32(p, B, st));
    } else {
      VSG_TRY(launch_cond(e.pre_w, e.pre_b, g, gp, H, e.gin, B, st));
    }
    gadd = gp;
  }
  if (y != x) VSG_CUDA_TRY(cudaMemcpyAsync(y, x, (size_t)n * sizeof(float), cudaMemcpyDeviceToDevice, st));
  relenc_addg_mask_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(y, gadd, g_t, mask, H, T, n);   // x = (x + g) * mask
  VSG_LAUNCH_CHECK("relenc_addg_mask_kernel");
  const unsigned ln_blocks = (unsigned)(((long long)B * T + 127) / 128);
  for (int i = 0; i < NL; ++i) {
    const RelEncLayer& L = e.layers[i];
    {  // q | k | v = conv_{q,k,v}(x)                                :124-126
      ConvF32 p = base_conv(L.qkv, y, HT, T, T, 0, 1);
      p.y = qkv; p.y_bs = 3 * HT; p.y_cs = T;
      VSG_TRY(launch_conv_f32(p, B, st));
    }
    VSG_TRY(attention_f32(dk, qkv, mask, L.ek, L.ev, o, B, e.n_heads, T, e.window, st));   // attention :137-177
    {  // x = x + conv_o(attn)                                        :130, :301
      ConvF32 p = base_conv(L.o, o, HT, T, T, 0, 1);
      p.res = y; p.res_bs = HT; p.res_cs = T;
      p.y = y; p.y_bs = HT; p.y_cs = T;
      VSG_TRY(launch_conv_f32(p, B, st));
    }
    relenc_layernorm_kernel<<<ln_blocks, 128, 0, st>>>(y, L.g1, L.b1, nullptr, 0, mask, 1e-4f, H, T, B);   // :303
    VSG_LAUNCH_CHECK("relenc_layernorm_kernel");
    {  // FFN: conv_1(x * mask) -> relu -> conv_2(. * mask)            :337-345
      ConvF32 p = base_conv(L.ffn1, y, HT, T, T, -(K / 2), 1);
      p.y = f; p.y_bs = (long long)F * T; p.y_cs = T; p.mask = mask; p.mask_bs = T;   // relu(h) * mask == relu(h * mask)
      VSG_TRY(launch_conv_f32(p, B, st));
    }
    {
      ConvF32 p = base_conv(L.ffn2, f, (long long)F * T, T, T, 0, 1);
      p.pre_lrelu = 1; p.slope = 0.f;                               // relu on load
      p.res = y; p.res_bs = HT; p.res_cs = T;
      p.y = y; p.y_bs = HT; p.y_cs = T;
      VSG_TRY(launch_conv_f32(p, B, st));
    }
    // x = LayerNorm(x); then the next layer's `x = (x + g) * mask` (:293-295) or the final `x * mask` (:318)
    relenc_layernorm_kernel<<<ln_blocks, 128, 0, st>>>(y, L.g2, L.b2, (i + 1 < NL) ? gadd : nullptr, g_t, mask, 1e-4f, H, T, B);
    VSG_LAUNCH_CHECK("relenc_layernorm_kernel");
  }
  return VSG_OK;
}

// FramePriorNetwork.forward (modules/visinger/encoder.py:67-73) + prior sampling (models/visinger.py:107), fp32 mode.
int frame_prior_forward_f32(const VsgPack* P, const float* x, const float* mask, const float* g, const float* noise,
                            float* stats, float* z, int B, int T, Workspace& ws, cudaStream_t st) {
  const RelEncPack& e = P->relenc;
  const int H = e.hidden;
  float* h = ws.take<float>((size_t)B * H * T);
  if (ws.overflow) return fail(VSG_ENOMEM, "frame prior workspace too small: need %zu bytes", ws.off);
  VSG_TRY(relenc_forward_f32(P, x, mask, g, g ? 1 : 0, h, B, T, ws, st));
  const size_t sm = (size_t)H * 32 * sizeof(float);
  dim3 grid((T + 31) / 32, B);
  prior_head_f32_kernel<<<grid, 256, sm, st>>>(h, e.proj_w, e.proj_b, noise, mask, stats, z, H, T);
  VSG_LAUNCH_CHECK("prior_head_f32_kernel");
  return VSG_OK;
}

int length_regulate(const float* enc, const long long* mel2ph, const float* table, int table_rows, float* y, int B, int H,
                    int T_ph, int T, cudaStream_t st) {
  length_regulate_pos_kernel<<<B, kLrThreads, 0, st>>>(enc, mel2ph, table, table_rows, y, H, T_ph, T);
  VSG_LAUNCH_CHECK("length_regulate_pos_kernel");
  return VSG_OK;
}

static size_t dec_max_elems(const VsgPack* P, int B, int T) {
  size_t m = (size_t)B * P->cfg.dec_upsample_initial_channel * T;
  long long L = T;
  for (const UpStage& st : P->ups) {
    L *= st.rate;
    m = std::max(m, (size_t)B * st.Cout * (size_t)L);
  }
  return m;
}

size_t dec_ws_bytes_f32(const VsgPack* P, int B, int T) {
  return align256((size_t)B * P->cfg.dec_upsample_initial_channel * sizeof(float)) +
         4 * align256(dec_max_elems(P, B, T) * sizeof(float));
}

// y [B, Cout, Lin * rate] = ConvTranspose1d(leaky_relu(x [B, Cin, Lin], 0.1)) + bias (decoder.py:45-46) as `rate` polyphase
// convolutions over the input rate, each writing every rate-th output sample.
int launch_upsample_f32(const UpStage& us, const float* x, int B, int Lin, float* y, cudaStream_t st) {
  const int Lout = Lin * us.rate;
  for (int r = 0; r < us.rate; ++r) {
    ConvF32 p = base_conv(us.phases[r].f32, x, (long long)us.Cin * Lin, Lin, Lin, us.phases[r].in_off0, 1);
    p.pre_lrelu = 1;
    p.Lq = (Lout - r + us.rate - 1) / us.rate; p.out_stride = us.rate; p.out_phase = r; p.Lout = Lout;
    p.y = y; p.y_bs = (long long)us.Cout * Lout; p.y_cs = Lout;
    VSG_TRY(launch_conv_f32(p, B, st));
  }
  return VSG_OK;
}

// wav = tanh(conv_post(leaky_relu(x [B, C, L], slope)))  (decoder.py:55-57; w [C][k] on the device, no bias): samples
// [n0, n1) of utterance b go to wav + b * wav_ld.
int launch_conv_post_f32(const float* x, const float* w, float* wav, int B, int C, int L, int k, float slope, int n0, int n1,
                         long long wav_ld, cudaStream_t st) {
  const size_t sm = (size_t)C * k * sizeof(float);
  if (sm > 48 * 1024) return fail(VSG_EUNSUPPORTED, "conv_post weights exceed 48 KB of shared memory (%zu B)", sm);
  if (n1 <= n0) return VSG_OK;
  dim3 grid((n1 - n0 + 255) / 256, B);
  conv_post_f32_kernel<<<grid, 256, sm, st>>>(x, w, wav, C, L, k, slope, n0, n1, wav_ld);
  VSG_LAUNCH_CHECK("conv_post_f32_kernel");
  return VSG_OK;
}

// Generator.forward, modules/visinger/decoder.py:40-59.
int generator_forward_f32(const VsgPack* P, const float* z, const float* g, float* wav, int B, int T, Workspace& ws,
                          cudaStream_t st, const DecWin* win) {
  const VsgConfig& c = P->cfg;
  const int UIC = c.dec_upsample_initial_channel, NK = c.dec_n_kernels;
  const size_t E = dec_max_elems(P, B, T);
  float* cond = ws.take<float>((size_t)B * UIC);
  float* bufS = ws.take<float>(E);   // stage input / running resblock sum
  float* bufU = ws.take<float>(E);   // upsampled x shared by the NK resblocks
  float* bufR = ws.take<float>(E);   // resblock running x
  float* bufT = ws.take<float>(E);   // conv1 output
  if (ws.overflow) return fail(VSG_ENOMEM, "generator workspace too small: need %zu bytes", ws.off);
  if (c.dec_gin > 0) {
    if (!g) return fail(VSG_EINVAL, "generator was built with gin_channels=%d but g is NULL", c.dec_gin);
    VSG_TRY(launch_cond(P->dec_cond_w, P->dec_cond_b, g, cond, UIC, c.dec_gin, B, st));
  }
  // x = conv_pre(z) + cond(g)                                        decoder.py:41-43
  {
    const int z_ld = win ? win->z_ld : T;
    ConvF32 p = base_conv(P->conv_pre, z, (long long)c.dec_initial_channel * z_ld, z_ld, T, -3, 1);
    if (c.dec_gin > 0) { p.bcond = cond; p.bcond_bs = UIC; }
    p.y = bufS; p.y_bs = (long long)UIC * T; p.y_cs = T;
    VSG_TRY(launch_conv_f32(p, B, st));
  }
  int L = T, ch = UIC;
  for (int i = 0; i < c.dec_n_ups; ++i) {
    const UpStage& us = P->ups[i];
    const int Lout = L * us.rate;
    VSG_TRY(launch_upsample_f32(us, bufS, B, L, bufU, st));   // x = ups[i](leaky_relu(x))   decoder.py:45-46
    ch = us.Cout; L = Lout;
    const long long bs = (long long)ch * L;
    // xs = sum_j resblock_j(x) ; x = xs / NK                           decoder.py:47-54
    for (int j = 0; j < NK; ++j) {
      const ResBlockPack& rb = us.blocks[j];
      const int nd = (int)rb.dilations.size();
      const int acc_mode = (j == 0) ? ACC_SET : (j == NK - 1 ? ACC_ADD_DIV : ACC_ADD);
      const float* cur = bufU;
      for (int q = 0; q < nd; ++q) {
        const bool last = (q == nd - 1);
        const int d = rb.dilations[q], k = rb.kernel;
        if (c.dec_resblock == 1) {   // ResBlock1, decoder.py:91-104
          ConvF32 p1 = base_conv(rb.c1[q], cur, bs, L, L, -((k * d - d) / 2), d);
          p1.pre_lrelu = 1; p1.y = bufT; p1.y_bs = bs; p1.y_cs = L;
          VSG_TRY(launch_conv_f32(p1, B, st));
          ConvF32 p2 = base_conv(rb.c2[q], bufT, bs, L, L, -((k - 1) / 2), 1);
          p2.pre_lrelu = 1; p2.res = cur; p2.res_bs = bs; p2.res_cs = L;
          p2.y = last ? bufS : bufR; p2.y_bs = bs; p2.y_cs = L;
          if (last) { p2.acc_mode = acc_mode; p2.acc_div = (float)NK; }
          VSG_TRY(launch_conv_f32(p2, B, st));
          cur = bufR;
        } else {                      // ResBlock2, decoder.py:124-133
          float* dst = last ? bufS : (cur == bufR ? bufT : bufR);
          ConvF32 p1 = base_conv(rb.c1[q], cur, bs, L, L, -((k * d - d) / 2), d);
          p1.pre_lrelu = 1; p1.res = cur; p1.res_bs = bs; p1.res_cs = L;
          p1.y = dst; p1.y_bs = bs; p1.y_cs = L;
          if (last) { p1.acc_mode = acc_mode; p1.acc_div = (float)NK; }
          VSG_TRY(launch_conv_f32(p1, B, st));
          cur = dst;
        }
      }
    }
    if (NK == 1) { /* xs / 1 == xs */ }
  }
  // wav = tanh(conv_post(leaky_relu(x)))                               decoder.py:55-57
  return launch_conv_post_f32(bufS, P->conv_post_w, wav, B, ch, L, P->conv_post_k, 0.1f, win ? win->s0 : 0,
                              win ? win->s1 : L, win ? win->wav_ld : (long long)L, st);
}

int prior_sample(const float* mu, const float* logs, const float* noise, const float* mask, float* z, int B, int C,
                 int T, cudaStream_t st) {
  const long long n = (long long)B * C * T;
  if (n == 0) return VSG_OK;
  prior_sample_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(mu, logs, noise, mask, z, C, T, n);
  VSG_LAUNCH_CHECK("prior_sample_kernel");
  return VSG_OK;
}

int mask_mul(const float* x, const float* mask, float* y, int B, int C, int T, cudaStream_t st, int mask_ld) {
  const long long n = (long long)B * C * T;
  if (n == 0) return VSG_OK;
  mask_mul_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x, mask, y, C, T, n, mask_ld > 0 ? mask_ld : T);
  VSG_LAUNCH_CHECK("mask_mul_kernel");
  return VSG_OK;
}

}  // namespace vsg

// Per-kernel parity hook of the fp32 attention kernel (tests only; synchronises).  See include/visinger_b200.h.
extern "C" int vsg_debug_attention_f32(const float* qkv, const float* mask, const float* ek, const float* ev, float* o,
                                       int32_t B, int32_t T, int32_t n_heads, int32_t dk, int32_t w, int32_t device) {
  using namespace vsg;
  reset_launch_counts();
  if (!qkv || !mask || !ek || !ev || !o) return fail(VSG_EINVAL, "null pointer");
  if (B < 1 || T < 1 || n_heads < 1 || w < 0) return fail(VSG_EINVAL, "bad argument");
  VSG_CUDA_TRY(cudaSetDevice(device));
  VSG_TRY(attention_f32(dk, qkv, mask, ek, ev, o, B, n_heads, T, w, 0));
  const cudaError_t ce = cudaDeviceSynchronize();
  if (ce != cudaSuccess) return fail(VSG_ECUDA, "relenc_attention_f32_kernel execution failed: %s", cudaGetErrorString(ce));
  return VSG_OK;
}

// One launch of conv_f32_kernel with every ConvF32 field (tests only; allocates and synchronises).  See include/visinger_b200.h.
extern "C" int vsg_debug_conv_f32(const VsgDebugConvF32* d, int32_t* tile_out, int32_t device) {
  using namespace vsg;
  reset_launch_counts();
  if (!d || !d->x || !d->w) return fail(VSG_EINVAL, "vsg_debug_conv_f32: null descriptor, input or weight");
  if (d->epi < EPI_LINEAR || d->epi > VSG_DEBUG_F32_MAG) return fail(VSG_EINVAL, "vsg_debug_conv_f32: epi must be 0 .. 4");
  if (d->B <= 0 || d->Cin <= 0 || d->Lin <= 0 || d->Cout <= 0 || d->k <= 0 || d->dil <= 0 || d->Lq <= 0 || d->Lout <= 0 ||
      d->out_stride <= 0 || d->out_phase < 0 || d->out_phase >= d->out_stride ||
      (long long)(d->Lq - 1) * d->out_stride + d->out_phase >= d->Lout)
    return fail(VSG_EINVAL, "vsg_debug_conv_f32: bad shape or output geometry");
  const bool pairs = d->epi == EPI_GATE || d->epi == VSG_DEBUG_F32_MAG;
  if (pairs && d->Cout % 2) return fail(VSG_EINVAL, "vsg_debug_conv_f32: gate and magnitude need an even Cout");
  if (d->gate_interleave && d->epi != EPI_GATE) return fail(VSG_EINVAL, "vsg_debug_conv_f32: gate_interleave is for the gate");
  if (d->x_cs < d->Lin || d->x_bs < (long long)d->Cin * d->x_cs)
    return fail(VSG_EINVAL, "vsg_debug_conv_f32: x rows overlap (x_cs < Lin or x_bs < Cin * x_cs)");
  if (d->mask && d->mask_bs < d->Lout) return fail(VSG_EINVAL, "vsg_debug_conv_f32: mask_bs < Lout");
  if (d->bcond && d->bcond_bs < d->Cout) return fail(VSG_EINVAL, "vsg_debug_conv_f32: bcond_bs < Cout");
  if (d->acc_mode < ACC_SET || d->acc_mode > ACC_ADD_DIV || (d->acc_mode != ACC_SET && d->epi != EPI_LINEAR) ||
      (d->acc_mode == ACC_ADD_DIV && d->acc_div == 0.f))
    return fail(VSG_EINVAL, "vsg_debug_conv_f32: acc_mode must be 0, 1 or 2 (linear only), acc_div nonzero");
  if (d->res && (d->epi != EPI_LINEAR && d->epi != EPI_COUPLE))
    return fail(VSG_EINVAL, "vsg_debug_conv_f32: res is read by the linear and couple epilogues only");
  if (d->res && (d->res_cs < d->Lout || d->res_bs < (long long)d->Cout * d->res_cs))
    return fail(VSG_EINVAL, "vsg_debug_conv_f32: res rows overlap (res_cs < Lout or res_bs < Cout * res_cs)");
  if (d->epi == EPI_COUPLE && d->couple_sign != 1 && d->couple_sign != -1)
    return fail(VSG_EINVAL, "vsg_debug_conv_f32: couple_sign must be +1 or -1");
  const bool rs = d->epi == EPI_RES_SKIP;
  if (rs && (d->rs_split < 0 || d->rs_split > d->Cout)) return fail(VSG_EINVAL, "vsg_debug_conv_f32: rs_split outside 0 .. Cout");
  const int y_ch = rs ? d->rs_split : pairs ? d->Cout / 2 : d->Cout, y2_ch = rs ? d->Cout - d->rs_split : 0;
  if (y_ch > 0 && (!d->y || d->y_cs < d->Lout || d->y_bs < (long long)y_ch * d->y_cs))
    return fail(VSG_EINVAL, "vsg_debug_conv_f32: y missing or its rows overlap");
  if (y2_ch > 0 && (!d->y2 || d->y2_cs < d->Lout || d->y2_bs < (long long)y2_ch * d->y2_cs))
    return fail(VSG_EINVAL, "vsg_debug_conv_f32: y2 missing or its rows overlap");
  DebugScope sc;
  VSG_TRY(sc.open(device));
  std::vector<float> W(d->w, d->w + (size_t)d->Cout * d->Cin * d->k), bz(d->Cout, 0.f);
  if (d->bias) bz.assign(d->bias, d->bias + d->Cout);
  ConvW32 wt;
  if (d->gate_interleave) VSG_TRY(pack_conv_f32(&sc.P, W, bz, d->Cout, d->Cin, d->k, GateInterleave{d->Cout / 2}, &wt));
  else VSG_TRY(pack_conv_f32(&sc.P, W, bz, d->Cout, d->Cin, d->k, Identity{}, &wt));
  ConvF32 p = base_conv(wt, d->x, d->x_bs, d->x_cs, d->Lin, d->in_off0, d->dil);
  p.pre_lrelu = d->pre_lrelu; p.slope = d->slope;
  p.bias = d->bias ? wt.bias : nullptr;
  p.bcond = d->bcond; p.bcond_bs = d->bcond_bs;
  p.Lq = d->Lq; p.out_stride = d->out_stride; p.out_phase = d->out_phase; p.Lout = d->Lout;
  p.epi = d->epi == VSG_DEBUG_F32_MAG ? EPI_LINEAR : d->epi;
  p.y = d->y; p.y_bs = d->y_bs; p.y_cs = d->y_cs;
  p.res = d->res; p.res_bs = d->res_bs; p.res_cs = d->res_cs;
  p.y2 = d->y2; p.y2_bs = d->y2_bs; p.y2_cs = d->y2_cs;
  p.mask = d->mask; p.mask_bs = d->mask_bs;
  p.acc_mode = d->acc_mode; p.acc_div = d->acc_div;
  p.rs_split = d->rs_split; p.y2_first = d->y2_first; p.y2_mask = d->y2_mask;
  p.couple_sign = d->couple_sign;
  int tile[2] = {0, 0};
  const int rc = d->epi == VSG_DEBUG_F32_MAG ? launch_conv_f32<true>(p, d->B, 0, tile) : launch_conv_f32(p, d->B, 0, tile);
  if (tile_out) { tile_out[0] = tile[0]; tile_out[1] = tile[1]; }
  return sc.finish(rc, "conv_f32_kernel");
}

// Host only: conv_f32_plan.  See include/visinger_b200.h.
extern "C" int vsg_debug_conv_f32_plan(int32_t Cout, int32_t k, int32_t dil, int32_t* out) {
  using namespace vsg;
  if (!out || Cout <= 0 || k <= 0 || dil <= 0) return fail(VSG_EINVAL, "vsg_debug_conv_f32_plan: bad argument");
  int wc = 0, wq = 0;
  size_t sm = 0;
  VSG_TRY(conv_f32_plan(Cout, k, dil, &wc, &wq, &sm));
  out[0] = wc; out[1] = wq; out[2] = (int32_t)sm;
  return VSG_OK;
}

// The decoder's upsampler as generator_forward_f32 runs it (tests only; allocates and synchronises).
extern "C" int vsg_debug_upsample_f32(const float* x, const float* w, const float* bias, int32_t Cin, int32_t Cout, int32_t rate,
                                      int32_t k, int32_t B, int32_t Lin, float* y, int32_t device) {
  using namespace vsg;
  reset_launch_counts();
  if (!x || !w || !bias || !y) return fail(VSG_EINVAL, "vsg_debug_upsample_f32: null input, weight, bias or output");
  if (Cin <= 0 || Cout <= 0 || B <= 0 || Lin <= 0 || rate <= 0 || k < rate || (k - rate) % 2)
    return fail(VSG_EINVAL, "vsg_debug_upsample_f32: bad shape (needs k >= rate and k - rate even)");
  if ((long long)Lin * rate >= (1LL << 31)) return fail(VSG_EINVAL, "vsg_debug_upsample_f32: output too long");
  DebugScope sc;
  VSG_TRY(sc.open(device));
  UpStage us;
  std::vector<float> W(w, w + (size_t)Cin * Cout * k), b(bias, bias + Cout);
  std::vector<std::vector<float>> phase_w;
  VSG_TRY(pack_upsampler(&sc.P, W, b, Cin, Cout, rate, k, &us, &phase_w));
  for (int r = 0; r < rate; ++r)
    VSG_TRY(pack_conv_f32(&sc.P, phase_w[r], b, Cout, Cin, (int)(phase_w[r].size() / ((size_t)Cout * Cin)), Identity{},
                          &us.phases[r].f32));
  return sc.finish(launch_upsample_f32(us, x, B, Lin, y, 0), "conv_f32_kernel");
}

// conv_post_f32_kernel through the generator's launcher (tests only; allocates and synchronises).
extern "C" int vsg_debug_conv_post_f32(const float* x, const float* w, int32_t C, int32_t L, int32_t k, float slope, int32_t B,
                                       int32_t n0, int32_t n1, float* wav, int64_t wav_ld, int32_t device) {
  using namespace vsg;
  reset_launch_counts();
  if (!x || !w || !wav) return fail(VSG_EINVAL, "vsg_debug_conv_post_f32: null input, weight or output");
  if (C <= 0 || L <= 0 || k <= 0 || B <= 0 || n0 < 0 || n1 <= n0 || n1 > L || wav_ld < n1 - n0)
    return fail(VSG_EINVAL, "vsg_debug_conv_post_f32: bad shape or window (needs 0 <= n0 < n1 <= L, wav_ld >= n1 - n0)");
  DebugScope sc;
  VSG_TRY(sc.open(device));
  float* dw = nullptr;
  VSG_TRY(upload(&sc.P, std::vector<float>(w, w + (size_t)C * k), &dw));
  return sc.finish(launch_conv_post_f32(x, dw, wav, B, C, L, k, slope, n0, n1, wav_ld, 0), "conv_post_f32_kernel");
}

// launch_cond (cond_gemv_kernel) (tests only; synchronises).
extern "C" int vsg_debug_cond_f32(const float* W, const float* bias, const float* g, float* out, int32_t O, int32_t I, int32_t B,
                                  int32_t device) {
  using namespace vsg;
  reset_launch_counts();
  if (!W || !g || !out) return fail(VSG_EINVAL, "vsg_debug_cond_f32: null weight, input or output");
  if (O <= 0 || I <= 0 || B <= 0 || (long long)O * B * 32 >= (1LL << 31))
    return fail(VSG_EINVAL, "vsg_debug_cond_f32: bad shape");
  DebugScope sc;
  VSG_TRY(sc.open(device));
  return sc.finish(launch_cond(W, bias, g, out, O, I, B, 0), "cond_gemv_kernel");
}
