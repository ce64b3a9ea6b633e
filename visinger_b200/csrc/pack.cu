// vsg_pack_create / vsg_pack_destroy: the one-time weight pre-pack.
//
// What the reference recomputes on every forward is folded here, once:
//   * weight-norm  w = v * (g / ||v||)   (torch.nn.utils.weight_norm pre-hook; applied at
//     modules/visinger/encoder.py:147,154,164 and modules/visinger/decoder.py:24-26,72-87,117-120);
//     for ConvTranspose1d the norm runs over dim 0 = C_in (SURVEY.md 7.2-7);
//   * Flip (modules/visinger/flow.py:88-95) -> channel-reversed copies of pre / post;
//   * the gate's tanh/sigmoid halves (encoder.py:206-213) -> interleaved output channels of
//     in_layers and cond_layer so one thread owns both halves of a channel;
//   * ConvTranspose1d -> `stride` polyphase dense sub-convolutions.
#include "vsg_common.cuh"
#include "pack_tc.cuh"

#include <math.h>
#include <algorithm>

namespace vsg {

thread_local char g_err[1024] = {0};
thread_local int g_launches = 0;
thread_local int g_image_launches[kImageSlots] = {0};

namespace {

struct HostTensor {
  const float* data;
  std::vector<int64_t> shape;
  int64_t numel() const { int64_t n = 1; for (auto s : shape) n *= s; return n; }
};

struct Loader {
  std::map<std::string, HostTensor> m;
  VsgPack* pack;

  const HostTensor* find(const std::string& k) const {
    auto it = m.find(k);
    return it == m.end() ? nullptr : &it->second;
  }

  // Effective weight of conv `prefix` as a flat vector in its stored [D0][D1][k] order.
  int eff_weight(const std::string& prefix, int64_t d0, int64_t d1, int64_t k, std::vector<float>& out) const {
    const int64_t n = d0 * d1 * k;
    out.resize(n);
    if (const HostTensor* w = find(prefix + ".weight")) {
      if (w->numel() != n) return fail(VSG_EINVAL, "%s.weight has %lld elements, expected %lld", prefix.c_str(),
                                       (long long)w->numel(), (long long)n);
      memcpy(out.data(), w->data, n * sizeof(float));
      return VSG_OK;
    }
    const HostTensor* g = find(prefix + ".weight_g");
    const HostTensor* v = find(prefix + ".weight_v");
    if (!g || !v) return fail(VSG_EINVAL, "missing weight for %s (.weight or .weight_g/.weight_v)", prefix.c_str());
    if (v->numel() != n || g->numel() != d0)
      return fail(VSG_EINVAL, "%s: weight_v has %lld elements (expected %lld), weight_g %lld (expected %lld)",
                  prefix.c_str(), (long long)v->numel(), (long long)n, (long long)g->numel(), (long long)d0);
    const int64_t inner = d1 * k;
    for (int64_t r = 0; r < d0; ++r) {
      double ss = 0.0;
      for (int64_t i = 0; i < inner; ++i) { double t = v->data[r * inner + i]; ss += t * t; }
      const float norm = (float)sqrt(ss);
      if (!(norm > 0.f))
        return fail(VSG_EINVAL, "%s.weight_v row %lld has zero norm: weight-norm w = g * v / ||v|| is undefined",
                    prefix.c_str(), (long long)r);
      const float scale = g->data[r] / norm;
      for (int64_t i = 0; i < inner; ++i) out[r * inner + i] = v->data[r * inner + i] * scale;
    }
    return VSG_OK;
  }

  int bias(const std::string& prefix, int64_t n, std::vector<float>& out, bool required) const {
    out.assign(n, 0.f);
    const HostTensor* b = find(prefix + ".bias");
    if (!b) return required ? fail(VSG_EINVAL, "missing %s.bias", prefix.c_str()) : VSG_OK;
    if (b->numel() != n) return fail(VSG_EINVAL, "%s.bias has %lld elements, expected %lld", prefix.c_str(),
                                     (long long)b->numel(), (long long)n);
    memcpy(out.data(), b->data, n * sizeof(float));
    return VSG_OK;
  }

  template <typename T>
  int upload(const std::vector<T>& h, T** d) const { return vsg::upload(pack, h, d); }
};

int pack_flow(const Loader& L, const std::string& pre, VsgPack* P) {
  const VsgConfig& c = P->cfg;
  const int C = c.flow_channels, H = c.flow_hidden, K = c.flow_kernel_size, NL = c.flow_n_layers, half = C / 2;
  if (C % 2 || C <= 0 || H <= 0 || NL <= 0 || K % 2 == 0 || c.flow_dilation_rate < 1)
    return fail(VSG_EINVAL, "bad flow config (channels %d hidden %d kernel %d layers %d)", C, H, K, NL);
  P->flow_layers.resize(c.flow_n_flows);
  std::vector<float> W, b, cond_w_all, cond_b_all;
  for (int f = 0; f < c.flow_n_flows; ++f) {
    FlowLayer& fl = P->flow_layers[f];
    const std::string p = pre + "flows." + std::to_string(2 * f) + ".";
    // pre: Conv1d(half -> H, 1)       flow.py:60
    VSG_TRY(L.eff_weight(p + "pre", H, half, 1, W));
    VSG_TRY(L.bias(p + "pre", H, b, true));
    VSG_TRY(pack_conv_f32(L.pack, W, b, H, half, 1, Identity{}, &fl.pre[0]));
    VSG_TRY(pack_conv_tc(P, W, b, H, half, 1, &fl.pre_tc[0]));
    VSG_TRY(pack_conv_tc(P, W, b, H, half, 1, &fl.pre_x6[0], 3));
    auto zero_extend = [&](const std::vector<float>& Wi, const std::vector<float>& bi, int flipped) -> int {
      std::vector<float> W2((size_t)2 * H * half, 0.f), b2((size_t)2 * H, 0.f);
      std::copy(Wi.begin(), Wi.end(), W2.begin());
      std::copy(bi.begin(), bi.end(), b2.begin());
      VSG_TRY(pack_conv_tc(P, W2, b2, 2 * H, half, 1, &fl.pre2_tc[flipped][0]));
      VSG_TRY(pack_conv_tc(P, W2, b2, 2 * H, half, 1, &fl.pre2_tc[flipped][1], 3));
      return VSG_OK;
    };
    VSG_TRY(zero_extend(W, b, 0));
    {
      std::vector<float> Wf(W.size());
      for (int co = 0; co < H; ++co)
        for (int ci = 0; ci < half; ++ci) Wf[(size_t)co * half + ci] = W[(size_t)co * half + (half - 1 - ci)];
      VSG_TRY(pack_conv_f32(L.pack, Wf, b, H, half, 1, Identity{}, &fl.pre[1]));
      VSG_TRY(pack_conv_tc(P, Wf, b, H, half, 1, &fl.pre_tc[1]));
      VSG_TRY(pack_conv_tc(P, Wf, b, H, half, 1, &fl.pre_x6[1], 3));
      VSG_TRY(zero_extend(Wf, b, 1));
    }
    // post: Conv1d(H -> half, 1)      flow.py:62 (mean_only)
    VSG_TRY(L.eff_weight(p + "post", half, H, 1, W));
    VSG_TRY(L.bias(p + "post", half, b, true));
    VSG_TRY(pack_conv_f32(L.pack, W, b, half, H, 1, Identity{}, &fl.post[0]));
    VSG_TRY(pack_conv_tc(P, W, b, half, H, 1, &fl.post_tc[0]));
    VSG_TRY(pack_conv_tc(P, W, b, half, H, 1, &fl.post_x6[0], 3));
    {
      std::vector<float> Wf(W.size()), bf(b.size());
      for (int co = 0; co < half; ++co) {
        bf[co] = b[half - 1 - co];
        for (int ci = 0; ci < H; ++ci) Wf[(size_t)co * H + ci] = W[(size_t)(half - 1 - co) * H + ci];
      }
      VSG_TRY(pack_conv_f32(L.pack, Wf, bf, half, H, 1, Identity{}, &fl.post[1]));
      VSG_TRY(pack_conv_tc(P, Wf, bf, half, H, 1, &fl.post_tc[1]));
      VSG_TRY(pack_conv_tc(P, Wf, bf, half, H, 1, &fl.post_x6[1], 3));
    }
    // WaveNet                        encoder.py:131-165
    fl.in_layers.resize(NL);
    fl.res_skip.resize(NL);
    fl.in_tc.resize(NL);
    fl.res_tc.resize(NL);
    fl.skip_tc.resize(NL);
    fl.in_x6.resize(NL); fl.res_x6.resize(NL); fl.skip_x6.resize(NL);
    fl.rs_tc[0].resize(NL); fl.rs_tc[1].resize(NL);
    for (int i = 0; i < NL; ++i) {
      const std::string pi = p + "enc.in_layers." + std::to_string(i);
      VSG_TRY(L.eff_weight(pi, 2 * H, H, K, W));
      VSG_TRY(L.bias(pi, 2 * H, b, true));
      VSG_TRY(pack_conv_f32(L.pack, W, b, 2 * H, H, K, GateInterleave{H}, &fl.in_layers[i]));
      {   // tensor-core pack: rows permuted so (tanh, sigmoid) halves of a channel sit in adjacent accumulator columns
        GateInterleave gi{H};
        std::vector<float> Wg(W.size()), bg(b.size());
        for (int co = 0; co < 2 * H; ++co) {
          bg[gi(co)] = b[co];
          memcpy(&Wg[(size_t)gi(co) * H * K], &W[(size_t)co * H * K], (size_t)H * K * sizeof(float));
        }
        VSG_TRY(pack_conv_tc(P, Wg, bg, 2 * H, H, K, &fl.in_tc[i]));
        VSG_TRY(pack_conv_tc(P, Wg, bg, 2 * H, H, K, &fl.in_x6[i], 3));
      }
      const int rs = (i < NL - 1) ? 2 * H : H;
      const std::string pr = p + "enc.res_skip_layers." + std::to_string(i);
      VSG_TRY(L.eff_weight(pr, rs, H, 1, W));
      VSG_TRY(L.bias(pr, rs, b, true));
      VSG_TRY(pack_conv_f32(L.pack, W, b, rs, H, 1, Identity{}, &fl.res_skip[i]));
      if (i < NL - 1) {
        VSG_TRY(pack_conv_tc(P, W, b, 2 * H, H, 1, &fl.rs_tc[0][i]));
        VSG_TRY(pack_conv_tc(P, W, b, 2 * H, H, 1, &fl.rs_tc[1][i], 3));
        std::vector<float> Wr(W.begin(), W.begin() + (size_t)H * H), br(b.begin(), b.begin() + H);
        std::vector<float> Ws(W.begin() + (size_t)H * H, W.end()), bs(b.begin() + H, b.end());
        VSG_TRY(pack_conv_tc(P, Wr, br, H, H, 1, &fl.res_tc[i]));
        VSG_TRY(pack_conv_tc(P, Wr, br, H, H, 1, &fl.res_x6[i], 3));
        VSG_TRY(pack_conv_tc(P, Ws, bs, H, H, 1, &fl.skip_tc[i]));
        VSG_TRY(pack_conv_tc(P, Ws, bs, H, H, 1, &fl.skip_x6[i], 3));
      } else {
        VSG_TRY(pack_conv_tc(P, W, b, H, H, 1, &fl.skip_tc[i]));
        VSG_TRY(pack_conv_tc(P, W, b, H, H, 1, &fl.skip_x6[i], 3));
      }
    }
    if (c.flow_gin > 0) {
      const int O = 2 * H * NL, I = c.flow_gin;
      VSG_TRY(L.eff_weight(p + "enc.cond_layer", O, I, 1, W));
      VSG_TRY(L.bias(p + "enc.cond_layer", O, b, true));
      std::vector<float> Wp(W.size()), bp(b.size());
      GateInterleave gi{H};
      for (int l = 0; l < NL; ++l)
        for (int cc = 0; cc < 2 * H; ++cc) {
          const int src = l * 2 * H + cc, dst = l * 2 * H + gi(cc);
          bp[dst] = b[src];
          memcpy(&Wp[(size_t)dst * I], &W[(size_t)src * I], I * sizeof(float));
        }
      VSG_TRY(L.upload(Wp, &fl.cond_w));
      VSG_TRY(L.upload(bp, &fl.cond_b));
      cond_w_all.insert(cond_w_all.end(), Wp.begin(), Wp.end());
      cond_b_all.insert(cond_b_all.end(), bp.begin(), bp.end());
    }
  }
  if (c.flow_gin > 0) {
    VSG_TRY(L.upload(cond_w_all, &P->flow_cond_w));
    VSG_TRY(L.upload(cond_b_all, &P->flow_cond_b));
  }
  P->has_flow = true;
  return VSG_OK;
}

// PosteriorEncoder: pre Conv1d(in -> H, 1), WaveNet(H, k, dilation_rate, n_layers, gin), proj Conv1d(H -> 2 out, 1)
// (modules/visinger/encoder.py:77-90; WaveNet layout encoder.py:131-165 as in pack_flow).
int pack_enc(const Loader& L, const std::string& p, VsgPack* P) {
  EncPack& e = P->enc;
  const int Cin = e.in_channels, Co = e.out_channels, H = e.hidden, K = e.kernel, NL = e.n_layers;
  if (Cin <= 0 || Co <= 0 || H <= 0 || NL <= 0 || K % 2 == 0 || e.dil_rate < 1 || e.gin < 0)
    return fail(VSG_EINVAL, "bad posterior encoder config (in %d out %d hidden %d kernel %d layers %d)", Cin, Co, H, K, NL);
  std::vector<float> W, b;
  VSG_TRY(L.eff_weight(p + "pre", H, Cin, 1, W));
  VSG_TRY(L.bias(p + "pre", H, b, true));
  VSG_TRY(pack_conv_f32(L.pack, W, b, H, Cin, 1, Identity{}, &e.pre));
  e.in_pad = round_up(Cin, 64);
  for (int c0 = 0; c0 < e.in_pad; c0 += 1024) {   // tensor-core packs: slabs of <= 1024 (zero-padded) input channels
    const int cs = std::min(1024, e.in_pad - c0);
    std::vector<float> Ws((size_t)H * cs, 0.f), bs(H, 0.f);
    for (int co = 0; co < H; ++co)
      for (int ci = 0; ci < cs && c0 + ci < Cin; ++ci) Ws[(size_t)co * cs + ci] = W[(size_t)co * Cin + c0 + ci];
    if (c0 == 0) bs = b;
    ConvWTC wt;
    VSG_TRY(pack_conv_tc(P, Ws, bs, H, cs, 1, &wt));
    e.pre_tc.push_back(wt);
    e.pre_c0.push_back(c0);
  }
  FlowLayer& fl = e.wn;
  fl.in_layers.resize(NL); fl.res_skip.resize(NL); fl.in_tc.resize(NL); fl.res_tc.resize(NL); fl.skip_tc.resize(NL);
  for (int i = 0; i < NL; ++i) {
    const std::string pi = p + "enc.in_layers." + std::to_string(i);
    VSG_TRY(L.eff_weight(pi, 2 * H, H, K, W));
    VSG_TRY(L.bias(pi, 2 * H, b, true));
    VSG_TRY(pack_conv_f32(L.pack, W, b, 2 * H, H, K, GateInterleave{H}, &fl.in_layers[i]));
    {
      GateInterleave gi{H};
      std::vector<float> Wg(W.size()), bg(b.size());
      for (int co = 0; co < 2 * H; ++co) {
        bg[gi(co)] = b[co];
        memcpy(&Wg[(size_t)gi(co) * H * K], &W[(size_t)co * H * K], (size_t)H * K * sizeof(float));
      }
      VSG_TRY(pack_conv_tc(P, Wg, bg, 2 * H, H, K, &fl.in_tc[i]));
    }
    const int rs = (i < NL - 1) ? 2 * H : H;
    const std::string pr = p + "enc.res_skip_layers." + std::to_string(i);
    VSG_TRY(L.eff_weight(pr, rs, H, 1, W));
    VSG_TRY(L.bias(pr, rs, b, true));
    VSG_TRY(pack_conv_f32(L.pack, W, b, rs, H, 1, Identity{}, &fl.res_skip[i]));
    if (i < NL - 1) {
      std::vector<float> Wr(W.begin(), W.begin() + (size_t)H * H), br(b.begin(), b.begin() + H);
      std::vector<float> Ws(W.begin() + (size_t)H * H, W.end()), bs(b.begin() + H, b.end());
      VSG_TRY(pack_conv_tc(P, Wr, br, H, H, 1, &fl.res_tc[i]));
      VSG_TRY(pack_conv_tc(P, Ws, bs, H, H, 1, &fl.skip_tc[i]));
    } else {
      VSG_TRY(pack_conv_tc(P, W, b, H, H, 1, &fl.skip_tc[i]));
    }
  }
  if (e.gin > 0) {
    const int O = 2 * H * NL, I = e.gin;
    VSG_TRY(L.eff_weight(p + "enc.cond_layer", O, I, 1, W));
    VSG_TRY(L.bias(p + "enc.cond_layer", O, b, true));
    std::vector<float> Wp(W.size()), bp(b.size());
    GateInterleave gi{H};
    for (int l = 0; l < NL; ++l)
      for (int cc = 0; cc < 2 * H; ++cc) {
        const int src = l * 2 * H + cc, dst = l * 2 * H + gi(cc);
        bp[dst] = b[src];
        memcpy(&Wp[(size_t)dst * I], &W[(size_t)src * I], I * sizeof(float));
      }
    VSG_TRY(L.upload(Wp, &fl.cond_w));
    VSG_TRY(L.upload(bp, &fl.cond_b));
  }
  VSG_TRY(L.eff_weight(p + "proj", 2 * Co, H, 1, W));
  VSG_TRY(L.bias(p + "proj", 2 * Co, b, true));
  VSG_TRY(pack_conv_f32(L.pack, W, b, 2 * Co, H, 1, Identity{}, &e.proj));
  VSG_TRY(pack_conv_tc(P, W, b, 2 * Co, H, 1, &e.proj_tc));
  P->has_enc = true;
  return VSG_OK;
}

// RelativeEncoder state-dict (modules/rel_transformer.py:272-284): attn_layers.N.{conv_q,conv_k,conv_v,conv_o}.{weight,bias},
// attn_layers.N.{emb_rel_k,emb_rel_v} [1][2w+1][dk], norm_layers_{1,2}.N.{gamma,beta}, ffn_layers.N.{conv_1,conv_2}.{weight,
// bias}, pre_net.{weight,bias}.  No weight-norm anywhere.
int pack_relenc(const Loader& L, const std::string& p, VsgPack* P, const char* proj_prefix = nullptr) {
  RelEncPack& e = P->relenc;
  const int H = e.hidden, F = e.filter, NL = e.n_layers, K = e.kernel, nh = e.n_heads, w = e.window;
  if (H <= 0 || F <= 0 || NL <= 0 || nh <= 0 || H % nh || K % 2 == 0 || w < 0 || w > 16)
    return fail(VSG_EINVAL, "bad encoder config (hidden %d filter %d heads %d layers %d kernel %d window %d)", H, F, nh, NL, K, w);
  const int dk = H / nh, nrel = 2 * w + 1;
  e.layers.resize(NL);
  std::vector<float> W, b, Wq, bq;
  auto vec = [&](const std::string& name, int64_t n, float** out) -> int {
    const HostTensor* t = L.find(name);
    if (!t || t->numel() != n) return fail(VSG_EINVAL, "missing or mis-shaped %s (expected %lld elements)", name.c_str(), (long long)n);
    std::vector<float> h(t->data, t->data + n);
    return L.upload(h, out);
  };
  for (int i = 0; i < NL; ++i) {
    RelEncLayer& l = e.layers[i];
    const std::string pa = p + "attn_layers." + std::to_string(i) + ".";
    Wq.assign((size_t)3 * H * H, 0.f); bq.assign((size_t)3 * H, 0.f);
    const char* names[3] = {"conv_q", "conv_k", "conv_v"};
    for (int s = 0; s < 3; ++s) {
      VSG_TRY(L.eff_weight(pa + names[s], H, H, 1, W));
      VSG_TRY(L.bias(pa + names[s], H, b, true));
      memcpy(&Wq[(size_t)s * H * H], W.data(), (size_t)H * H * sizeof(float));
      memcpy(&bq[(size_t)s * H], b.data(), (size_t)H * sizeof(float));
    }
    VSG_TRY(pack_conv_f32(L.pack, Wq, bq, 3 * H, H, 1, Identity{}, &l.qkv));
    VSG_TRY(pack_conv_tc(P, Wq, bq, 3 * H, H, 1, &l.qkv_tc));
    VSG_TRY(L.eff_weight(pa + "conv_o", H, H, 1, W));
    VSG_TRY(L.bias(pa + "conv_o", H, b, true));
    VSG_TRY(pack_conv_f32(L.pack, W, b, H, H, 1, Identity{}, &l.o));
    VSG_TRY(pack_conv_tc(P, W, b, H, H, 1, &l.o_tc));
    VSG_TRY(vec(pa + "emb_rel_k", (int64_t)nrel * dk, &l.ek));      // heads_share = True: [1][2w+1][dk]
    VSG_TRY(vec(pa + "emb_rel_v", (int64_t)nrel * dk, &l.ev));
    const std::string pf = p + "ffn_layers." + std::to_string(i) + ".";
    VSG_TRY(L.eff_weight(pf + "conv_1", F, H, K, W));
    VSG_TRY(L.bias(pf + "conv_1", F, b, true));
    VSG_TRY(pack_conv_f32(L.pack, W, b, F, H, K, Identity{}, &l.ffn1));
    VSG_TRY(pack_conv_tc(P, W, b, F, H, K, &l.ffn1_tc));
    VSG_TRY(L.eff_weight(pf + "conv_2", H, F, 1, W));
    VSG_TRY(L.bias(pf + "conv_2", H, b, true));
    VSG_TRY(pack_conv_f32(L.pack, W, b, H, F, 1, Identity{}, &l.ffn2));
    VSG_TRY(pack_conv_tc(P, W, b, H, F, 1, &l.ffn2_tc));
    VSG_TRY(vec(p + "norm_layers_1." + std::to_string(i) + ".gamma", H, &l.g1));
    VSG_TRY(vec(p + "norm_layers_1." + std::to_string(i) + ".beta", H, &l.b1));
    VSG_TRY(vec(p + "norm_layers_2." + std::to_string(i) + ".gamma", H, &l.g2));
    VSG_TRY(vec(p + "norm_layers_2." + std::to_string(i) + ".beta", H, &l.b2));
  }
  if (e.gin > 0) {
    VSG_TRY(L.eff_weight(p + "pre_net", H, e.gin, 1, W));
    VSG_TRY(L.bias(p + "pre_net", H, b, true));
    VSG_TRY(pack_conv_f32(L.pack, W, b, H, e.gin, 1, Identity{}, &e.pre_net));
    VSG_TRY(L.upload(W, &e.pre_w));
    VSG_TRY(L.upload(b, &e.pre_b));
  }
  if (proj_prefix) {   // FramePriorNetwork.proj: Conv1d(H -> 2H, 1)      modules/visinger/encoder.py:65
    const std::string pp = std::string(proj_prefix) + "proj";
    VSG_TRY(L.eff_weight(pp, 2 * H, H, 1, W));
    VSG_TRY(L.bias(pp, 2 * H, b, true));
    VSG_TRY(L.upload(W, &e.proj_w));
    VSG_TRY(L.upload(b, &e.proj_b));
    VSG_TRY(pack_conv_tc(P, W, b, 2 * H, H, 1, &e.proj_tc));
  }
  P->has_relenc = true;
  return VSG_OK;
}

int pack_decoder(const Loader& L, const std::string& pre, VsgPack* P) {
  const VsgConfig& c = P->cfg;
  const int C0 = c.dec_initial_channel, UIC = c.dec_upsample_initial_channel;
  if (c.dec_n_ups > VSG_MAX_UPS || c.dec_n_kernels > VSG_MAX_RESBLOCK_KERNELS || c.dec_n_kernels <= 0 ||
      (c.dec_resblock != 1 && c.dec_resblock != 2) || C0 <= 0 || UIC <= 0 || (UIC >> c.dec_n_ups) <= 0)
    return fail(VSG_EINVAL, "bad decoder config");
  std::vector<float> W, b;
  // conv_pre: Conv1d(C0 -> UIC, 7, padding 3), no weight norm   decoder.py:19
  VSG_TRY(L.eff_weight(pre + "conv_pre", UIC, C0, 7, W));
  VSG_TRY(L.bias(pre + "conv_pre", UIC, b, true));
  VSG_TRY(pack_conv_f32(L.pack, W, b, UIC, C0, 7, Identity{}, &P->conv_pre));
  VSG_TRY(pack_conv_tc(P, W, b, UIC, C0, 7, &P->conv_pre_tc));
  VSG_TRY(pack_conv_tc(P, W, b, UIC, C0, 7, &P->conv_pre_x3, 2));
  if (c.dec_gin > 0) {   // cond: Conv1d(gin -> UIC, 1)            decoder.py:37-38
    VSG_TRY(L.eff_weight(pre + "cond", UIC, c.dec_gin, 1, W));
    VSG_TRY(L.bias(pre + "cond", UIC, b, true));
    VSG_TRY(L.upload(W, &P->dec_cond_w));
    VSG_TRY(L.upload(b, &P->dec_cond_b));
  }
  P->ups.resize(c.dec_n_ups);
  P->hop = 1;
  int ch = UIC;
  for (int i = 0; i < c.dec_n_ups; ++i) {
    UpStage& st = P->ups[i];
    st.rate = c.dec_upsample_rates[i];
    st.kernel = c.dec_upsample_kernel_sizes[i];
    st.Cin = UIC >> i;
    st.Cout = UIC >> (i + 1);
    st.pad = (st.kernel - st.rate) / 2;
    if (st.rate < 1 || st.kernel < st.rate || (st.kernel - st.rate) % 2)
      return fail(VSG_EUNSUPPORTED, "ups.%d: kernel %d / stride %d needs kernel >= stride and (kernel - stride) even",
                  i, st.kernel, st.rate);
    P->hop *= st.rate;
    ch = st.Cout;
    // ConvTranspose1d weight [Cin][Cout][k], weight-norm over dim 0 = Cin   decoder.py:24-26
    const std::string pu = pre + "ups." + std::to_string(i);
    VSG_TRY(L.eff_weight(pu, st.Cin, st.Cout, st.kernel, W));
    VSG_TRY(L.bias(pu, st.Cout, b, true));
    std::vector<std::vector<float>> phase_w;
    VSG_TRY(pack_upsampler(P, W, b, st.Cin, st.Cout, st.rate, st.kernel, &st, &phase_w));
    for (int r = 0; r < st.rate; ++r)
      VSG_TRY(pack_conv_f32(L.pack, phase_w[r], b, st.Cout, st.Cin, (int)(phase_w[r].size() / ((size_t)st.Cout * st.Cin)), Identity{},
                            &st.phases[r].f32));
    // resblocks                                                            decoder.py:28-32
    st.blocks.resize(c.dec_n_kernels);
    for (int j = 0; j < c.dec_n_kernels; ++j) {
      ResBlockPack& rb = st.blocks[j];
      rb.kernel = c.dec_resblock_kernel_sizes[j];
      if (rb.kernel % 2 == 0) return fail(VSG_EUNSUPPORTED, "even resblock kernel size %d", rb.kernel);
      const int nd = c.dec_n_dilations[j];
      if (nd <= 0 || nd > VSG_MAX_RESBLOCK_DILATIONS) return fail(VSG_EINVAL, "bad dilation count");
      rb.dilations.assign(c.dec_resblock_dilations[j], c.dec_resblock_dilations[j] + nd);
      const std::string pb = pre + "resblocks." + std::to_string(i * c.dec_n_kernels + j) + ".";
      rb.c1.resize(nd); rb.c1_tc.resize(nd); rb.c1_x3.resize(nd);
      if (c.dec_resblock == 1) { rb.c2.resize(nd); rb.c2_tc.resize(nd); rb.c2_x3.resize(nd); rb.c1_rp.resize(nd); rb.c2_rp.resize(nd);
                                   rb.c1_rp_x3.resize(nd); rb.c2_rp_x3.resize(nd); }
      std::vector<std::vector<float>> b2s;
      for (int q = 0; q < nd; ++q) {
        const std::string n1 = pb + (c.dec_resblock == 1 ? "convs1." : "convs.") + std::to_string(q);
        VSG_TRY(L.eff_weight(n1, ch, ch, rb.kernel, W));
        VSG_TRY(L.bias(n1, ch, b, true));
        VSG_TRY(pack_conv_f32(L.pack, W, b, ch, ch, rb.kernel, Identity{}, &rb.c1[q]));
        VSG_TRY(pack_conv_tc(P, W, b, ch, ch, rb.kernel, &rb.c1_tc[q]));
        VSG_TRY(pack_conv_tc(P, W, b, ch, ch, rb.kernel, &rb.c1_x3[q], 2));
        if (c.dec_resblock == 1 && rb.dilations[q] == 1) {
          VSG_TRY(pack_conv_rowpacked(P, W, ch, rb.kernel, &rb.c1_rp[q]));
          VSG_TRY(pack_conv_rowpacked(P, W, ch, rb.kernel, &rb.c1_rp_x3[q], 2));
        }
        if (c.dec_resblock == 1) {
          const std::string n2 = pb + "convs2." + std::to_string(q);
          VSG_TRY(L.eff_weight(n2, ch, ch, rb.kernel, W));
          VSG_TRY(L.bias(n2, ch, b, true));
          VSG_TRY(pack_conv_f32(L.pack, W, b, ch, ch, rb.kernel, Identity{}, &rb.c2[q]));
          VSG_TRY(pack_conv_tc(P, W, b, ch, ch, rb.kernel, &rb.c2_tc[q]));
          VSG_TRY(pack_conv_tc(P, W, b, ch, ch, rb.kernel, &rb.c2_x3[q], 2));
          VSG_TRY(pack_conv_rowpacked(P, W, ch, rb.kernel, &rb.c2_rp[q]));
          VSG_TRY(pack_conv_rowpacked(P, W, ch, rb.kernel, &rb.c2_rp_x3[q], 2));
          b2s.push_back(b);
        }
      }
      if (c.dec_resblock == 1 && ch <= 64) VSG_TRY(pack_resblock_bias_sums(P, b2s, &rb));
    }
  }
  // conv_post: Conv1d(ch -> 1, 7, padding 3, bias=False)                    decoder.py:34
  VSG_TRY(L.eff_weight(pre + "conv_post", 1, ch, 7, W));
  VSG_TRY(L.upload(W, &P->conv_post_w));
  P->conv_post_k = 7;
  // Tensor-core form (plain bf16 mode): S = 64 / ch consecutive samples are one 128-byte row of the channels-last stage
  // output, and conv_post becomes Conv1d(64 -> 16, 3 row taps) with block-Toeplitz weights whose output column s' < S is
  // sample S r + s' of row r:   W'[s'][s ch + c][m] = w[c][S (m - 1) + s - s' + 3]   (zero outside the 7 taps).
  if ((ch == 16 || ch == 32) && 64 / ch >= 3) {
    const int S = 64 / ch;
    std::vector<float> Wt((size_t)16 * 64 * 3, 0.f), bz(16, 0.f);
    for (int sp = 0; sp < S; ++sp)
      for (int m = 0; m < 3; ++m)
        for (int s2 = 0; s2 < S; ++s2) {
          const int j = S * (m - 1) + s2 - sp + 3;
          if (j < 0 || j >= 7) continue;
          for (int cc = 0; cc < ch; ++cc) Wt[((size_t)sp * 64 + s2 * ch + cc) * 3 + m] = W[(size_t)cc * 7 + j];
        }
    VSG_TRY(pack_conv_tc(P, Wt, bz, 16, 64, 3, &P->conv_post_rp, 2));   // [W_hi | W_lo]: no weight rounding in the last layer
    P->conv_post_rp.wsplit = true;
    if (P->conv_post_rp.has_tmap) P->conv_post_S = S;
  }
  // bf16x3 mode: a sample of the stage output is [hi (ch) | lo (ch)] = 2 ch bf16, so 64 / (2 ch) samples make a row and the
  // "input channels" of the row-packed convolution are (sample, plane, channel); both planes meet the same weights.
  if (ch == 16) {
    const int S = 2, RT = 5;       // rows r-2 .. r+2 cover samples 2r-4 .. 2r+5 (taps reach 2r-3 .. 2r+4)
    std::vector<float> Wt((size_t)16 * 64 * RT, 0.f), bz(16, 0.f);
    for (int sp = 0; sp < S; ++sp)
      for (int m = 0; m < RT; ++m)
        for (int s2 = 0; s2 < S; ++s2) {
          const int j = S * (m - 2) + s2 - sp + 3;
          if (j < 0 || j >= 7) continue;
          for (int pl = 0; pl < 2; ++pl)
            for (int cc = 0; cc < ch; ++cc)
              Wt[((size_t)sp * 64 + s2 * 2 * ch + pl * ch + cc) * RT + m] = W[(size_t)cc * 7 + j];
        }
    VSG_TRY(pack_conv_tc(P, Wt, bz, 16, 64, RT, &P->conv_post_rp_x3, 2));
    P->conv_post_rp_x3.wsplit = true;
  }
  P->has_dec = true;
  return VSG_OK;
}

}  // namespace
}  // namespace vsg

using namespace vsg;

extern "C" int vsg_abi_version(void) { return VSG_ABI_VERSION; }
extern "C" const char* vsg_last_error(void) { return vsg::g_err; }
extern "C" int32_t vsg_last_launch_count(void) { return vsg::g_launches; }
extern "C" int vsg_last_launch_images(int32_t* out, int32_t n) {
  if (!out || n < 0) return vsg::fail(VSG_EINVAL, "vsg_last_launch_images: null output or negative count");
  for (int32_t i = 0; i < n; ++i) out[i] = i < vsg::kImageSlots ? vsg::g_image_launches[i] : 0;
  return VSG_OK;
}
extern "C" int32_t vsg_hop_size(const VsgPack* p) {
  if (p && p->model) p = p->model->hot;
  return (p && p->has_dec) ? p->hop : 0;
}

extern "C" int vsg_pack_create(const VsgConfig* cfg, const VsgTensor* weights, int32_t n_weights,
                               const char* flow_prefix, const char* dec_prefix, int32_t device, VsgPack** out) {
  if (!cfg || !out || (!weights && n_weights > 0)) return fail(VSG_EINVAL, "null argument");
  *out = nullptr;
  int ndev = 0;
  VSG_CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(VSG_EINVAL, "device %d out of range (%d visible)", device, ndev);
  // every exit below restores the caller's current device
  struct Restore { int prev = -1; ~Restore() { if (prev >= 0) cudaSetDevice(prev); } } restore;
  VSG_CUDA_TRY(cudaGetDevice(&restore.prev));
  VSG_CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  VSG_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(VSG_EUNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device,
                prop.major, prop.minor);
  VsgPack* P = new VsgPack();
  P->cfg = *cfg;
  P->device = device;
  P->sm_count = prop.multiProcessorCount;
  Loader L;
  L.pack = P;
  for (int i = 0; i < n_weights; ++i) {
    if (!weights[i].name || !weights[i].data || weights[i].ndim < 0 || weights[i].ndim > 4) {
      delete P;
      return fail(VSG_EINVAL, "weight table entry %d is malformed", i);
    }
    HostTensor t;
    t.data = weights[i].data;
    t.shape.assign(weights[i].shape, weights[i].shape + weights[i].ndim);
    L.m[weights[i].name] = t;
  }
  int rc = VSG_OK;
  if (cfg->flow_n_flows > 0) rc = pack_flow(L, flow_prefix ? flow_prefix : "", P);
  if (rc == VSG_OK && cfg->dec_n_ups > 0) rc = pack_decoder(L, dec_prefix ? dec_prefix : "", P);
  if (rc == VSG_OK && !P->has_flow && !P->has_dec) rc = fail(VSG_EINVAL, "config selects neither flow nor decoder");
  if (rc != VSG_OK) {
    vsg_pack_destroy(P);
    return rc;
  }
  *out = P;
  return VSG_OK;
}

extern "C" int vsg_enc_pack_create(const VsgEncConfig* cfg, const VsgTensor* weights, int32_t n_weights, const char* prefix,
                                   int32_t device, VsgPack** out) {
  if (!cfg || !out || (!weights && n_weights > 0)) return fail(VSG_EINVAL, "null argument");
  *out = nullptr;
  int ndev = 0;
  VSG_CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(VSG_EINVAL, "device %d out of range (%d visible)", device, ndev);
  struct Restore { int prev = -1; ~Restore() { if (prev >= 0) cudaSetDevice(prev); } } restore;
  VSG_CUDA_TRY(cudaGetDevice(&restore.prev));
  VSG_CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  VSG_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(VSG_EUNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device,
                prop.major, prop.minor);
  VsgPack* P = new VsgPack();
  memset(&P->cfg, 0, sizeof(P->cfg));
  P->device = device;
  P->sm_count = prop.multiProcessorCount;
  P->enc.in_channels = cfg->in_channels; P->enc.out_channels = cfg->out_channels; P->enc.hidden = cfg->hidden_channels;
  P->enc.kernel = cfg->kernel_size; P->enc.dil_rate = cfg->dilation_rate; P->enc.n_layers = cfg->n_layers;
  P->enc.gin = cfg->gin_channels;
  Loader L;
  L.pack = P;
  for (int i = 0; i < n_weights; ++i) {
    if (!weights[i].name || !weights[i].data || weights[i].ndim < 0 || weights[i].ndim > 4) {
      delete P;
      return fail(VSG_EINVAL, "weight table entry %d is malformed", i);
    }
    HostTensor t;
    t.data = weights[i].data;
    t.shape.assign(weights[i].shape, weights[i].shape + weights[i].ndim);
    L.m[weights[i].name] = t;
  }
  const int rc = pack_enc(L, prefix ? prefix : "", P);
  if (rc != VSG_OK) {
    vsg_pack_destroy(P);
    return rc;
  }
  *out = P;
  return VSG_OK;
}

static int relenc_pack_create(const VsgRelEncConfig* cfg, const VsgTensor* weights, int32_t n_weights, const char* prefix,
                              const char* proj_prefix, int32_t device, VsgPack** out);

extern "C" int vsg_relenc_pack_create(const VsgRelEncConfig* cfg, const VsgTensor* weights, int32_t n_weights,
                                      const char* prefix, int32_t device, VsgPack** out) {
  return relenc_pack_create(cfg, weights, n_weights, prefix, nullptr, device, out);
}

extern "C" int vsg_frame_prior_pack_create(const VsgRelEncConfig* cfg, const VsgTensor* weights, int32_t n_weights,
                                           const char* prefix, int32_t device, VsgPack** out) {
  const std::string p = prefix ? prefix : "";
  return relenc_pack_create(cfg, weights, n_weights, (p + "encoder.").c_str(), p.c_str(), device, out);
}

static int relenc_pack_create(const VsgRelEncConfig* cfg, const VsgTensor* weights, int32_t n_weights, const char* prefix,
                              const char* proj_prefix, int32_t device, VsgPack** out) {
  if (!cfg || !out || (!weights && n_weights > 0)) return fail(VSG_EINVAL, "null argument");
  *out = nullptr;
  int ndev = 0;
  VSG_CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(VSG_EINVAL, "device %d out of range (%d visible)", device, ndev);
  struct Restore { int prev = -1; ~Restore() { if (prev >= 0) cudaSetDevice(prev); } } restore;
  VSG_CUDA_TRY(cudaGetDevice(&restore.prev));
  VSG_CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  VSG_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(VSG_EUNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device,
                prop.major, prop.minor);
  VsgPack* P = new VsgPack();
  memset(&P->cfg, 0, sizeof(P->cfg));
  P->device = device;
  P->sm_count = prop.multiProcessorCount;
  RelEncPack& e = P->relenc;
  e.hidden = cfg->hidden_channels; e.filter = cfg->filter_channels; e.n_heads = cfg->n_heads; e.n_layers = cfg->n_layers;
  e.kernel = cfg->kernel_size; e.window = cfg->window_size; e.gin = cfg->gin_channels;
  Loader L;
  L.pack = P;
  for (int i = 0; i < n_weights; ++i) {
    if (!weights[i].name || !weights[i].data || weights[i].ndim < 0 || weights[i].ndim > 4) {
      delete P;
      return fail(VSG_EINVAL, "weight table entry %d is malformed", i);
    }
    HostTensor t;
    t.data = weights[i].data;
    t.shape.assign(weights[i].shape, weights[i].shape + weights[i].ndim);
    L.m[weights[i].name] = t;
  }
  const int rc = pack_relenc(L, prefix ? prefix : "", P, proj_prefix);
  if (rc != VSG_OK) {
    vsg_pack_destroy(P);
    return rc;
  }
  *out = P;
  return VSG_OK;
}

extern "C" void vsg_pack_destroy(VsgPack* pack) {
  if (!pack) return;
  if (pack->model) vsg::model_pack_free(pack->model);
  int prev = 0;
  cudaGetDevice(&prev);
  cudaSetDevice(pack->device);
  for (void* p : pack->allocs) cudaFree(p);
  cudaSetDevice(prev);
  delete pack;
}
