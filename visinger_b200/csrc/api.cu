// extern "C" entry points of include/visinger_b200.h: argument validation and dispatch.
#include "vsg_common.cuh"
#include "run.cuh"

using namespace vsg;

namespace {

int check_common(const VsgPack* pack, int B, int T, int precision) {
  if (!pack) return fail(VSG_EINVAL, "pack is NULL");
  if (B < 0 || T < 0) return fail(VSG_EINVAL, "negative batch (%d) or length (%d)", B, T);
  if (B > 65535) return fail(VSG_EUNSUPPORTED, "batch %d exceeds 65535", B);
  if (precision != VSG_PRECISION_FP32 && precision != VSG_PRECISION_BF16 && precision != VSG_PRECISION_BF16X3)
    return fail(VSG_EINVAL, "unknown precision %d", precision);
  return VSG_OK;
}

}  // namespace

namespace vsg {

size_t flow_ws(const VsgPack* p, int B, int T, int prec) {
  if (!p->has_flow) return 0;
  if (prec == VSG_PRECISION_BF16) return flow_ws_bytes_tc(p, B, T, 1);
  if (prec == VSG_PRECISION_BF16X3) return std::max(flow_ws_bytes_tc(p, B, T, 3), flow_ws_bytes_f32(p, B, T));
  return flow_ws_bytes_f32(p, B, T);
}
size_t dec_ws(const VsgPack* p, int B, int T, int prec) {
  if (!p->has_dec) return 0;
  return prec == VSG_PRECISION_FP32 ? dec_ws_bytes_f32(p, B, T) : dec_ws_bytes_tc(p, B, T, prec == VSG_PRECISION_BF16X3);
}

// fp32: CUDA-core FFMA kernels.  bf16: tcgen05, one bf16 plane.  bf16x3: tcgen05 on three bf16 planes per value (the
// flow's z <= 1e-5 needs all 24 mantissa bits of its state; the decoder's 1e-4 is met by two planes).
// *masked (optional): in = the caller wants y * mask; out = true if the flow's last kernel applied it (tensor-core modes:
// the mask rides on the final layout change), false if the caller still has to
int run_flow(const VsgPack* pack, const float* x, const float* mask, const float* g, float* y, int B, int T, int reverse,
             int precision, Workspace& ws, cudaStream_t st, bool* masked, const float* ps_logs, const float* ps_noise,
             bool* sampled, int x_ld) {
  // ps_logs / ps_noise (with `sampled`): x is mu_p; *sampled = true if the flow's first kernel drew the prior sample itself
  if (sampled) *sampled = false;
  const bool want = masked && *masked;
  if (masked) *masked = false;
  const bool tc1 = precision == VSG_PRECISION_BF16;
  const bool tc3 = precision == VSG_PRECISION_BF16X3 && x3_flow_on_tensor_cores() && !pack->flow_layers.empty() &&
                   pack->flow_layers[0].pre_x6[0].has_tmap;
  if (tc1 || tc3) {
    if (masked) *masked = want;
    if (sampled && ps_logs && ps_noise) *sampled = true;
    return flow_forward_tc(pack, x, mask, g, y, B, T, reverse, ws, st, tc1 ? 1 : 3, want ? mask : nullptr,
                           sampled ? ps_logs : nullptr, sampled ? ps_noise : nullptr, x_ld);
  }
  return flow_forward_f32(pack, x, mask, g, y, B, T, reverse, ws, st, x_ld);
}

}  // namespace vsg

extern "C" size_t vsg_workspace_bytes(const VsgPack* pack, int32_t B, int32_t T, int32_t precision) {
  if (check_common(pack, B, T, precision) != VSG_OK) return 0;
  const size_t z = pack->has_flow ? align256((size_t)B * pack->cfg.flow_channels * T * sizeof(float))
                                  : align256((size_t)B * pack->cfg.dec_initial_channel * T * sizeof(float));
  return z + std::max(flow_ws(pack, B, T, precision), dec_ws(pack, B, T, precision)) + 1024;
}

extern "C" int vsg_prior_sample(const float* mu_p, const float* logs_p, const float* noise, const float* mask,
                                float* z_p, int32_t B, int32_t C, int32_t T, void* stream) {
  reset_launch_counts();
  if (B < 0 || C < 0 || T < 0) return fail(VSG_EINVAL, "negative dimension");
  if ((long long)B * C * T == 0) return VSG_OK;
  if (!mu_p || !logs_p || !noise || !mask || !z_p) return fail(VSG_EINVAL, "null pointer");
  return prior_sample(mu_p, logs_p, noise, mask, z_p, B, C, T, (cudaStream_t)stream);
}

extern "C" int vsg_flow_forward(const VsgPack* pack, const float* x, const float* mask, const float* g, float* y,
                                int32_t B, int32_t T, int32_t reverse, int32_t precision, void* workspace,
                                size_t workspace_bytes, void* stream) {
  reset_launch_counts();
  VSG_TRY(check_common(pack, B, T, precision));
  if (!pack->has_flow) return fail(VSG_EINVAL, "pack has no flow");
  if (B == 0 || T == 0) return VSG_OK;
  if (!x || !mask || !y) return fail(VSG_EINVAL, "null pointer");
  if (!workspace) return fail(VSG_ENOMEM, "workspace is NULL");
  DeviceGuard dg(pack->device);
  if (!dg.ok) return fail(VSG_ECUDA, "cannot select device %d", pack->device);
  Workspace ws(workspace, workspace_bytes);
  return run_flow(pack, x, mask, g, y, B, T, reverse, precision, ws, (cudaStream_t)stream);
}

extern "C" int vsg_generator_forward(const VsgPack* pack, const float* z, const float* g, float* wav, int32_t B,
                                     int32_t T, int32_t precision, void* workspace, size_t workspace_bytes,
                                     void* stream) {
  reset_launch_counts();
  VSG_TRY(check_common(pack, B, T, precision));
  if (!pack->has_dec) return fail(VSG_EINVAL, "pack has no decoder");
  if (B == 0 || T == 0) return VSG_OK;
  if (!z || !wav) return fail(VSG_EINVAL, "null pointer");
  if (!workspace) return fail(VSG_ENOMEM, "workspace is NULL");
  if ((long long)T * pack->hop > 0x7fffffffLL / 4) return fail(VSG_EUNSUPPORTED, "sequence too long (%d frames)", T);
  DeviceGuard dg(pack->device);
  if (!dg.ok) return fail(VSG_ECUDA, "cannot select device %d", pack->device);
  Workspace ws(workspace, workspace_bytes);
  if (precision == VSG_PRECISION_FP32)
    return generator_forward_f32(pack, z, g, wav, B, T, ws, (cudaStream_t)stream);
  return generator_forward_tc(pack, z, g, wav, B, T, ws, (cudaStream_t)stream, precision == VSG_PRECISION_BF16X3);
}

extern "C" int vsg_infer(const VsgPack* pack, const float* mu_p, const float* logs_p, const float* noise,
                         const float* mask, const float* g, float* wav, float* z_q_out, int32_t B, int32_t T,
                         int32_t precision, void* workspace, size_t workspace_bytes, void* stream) {
  reset_launch_counts();
  VSG_TRY(check_common(pack, B, T, precision));
  if (!pack->has_flow || !pack->has_dec) return fail(VSG_EINVAL, "vsg_infer needs a pack with both flow and decoder");
  if (pack->cfg.flow_channels != pack->cfg.dec_initial_channel)
    return fail(VSG_EINVAL, "flow channels (%d) != decoder initial_channel (%d)", pack->cfg.flow_channels,
                pack->cfg.dec_initial_channel);
  if (B == 0 || T == 0) return VSG_OK;
  if (!mu_p || !logs_p || !noise || !mask || !wav) return fail(VSG_EINVAL, "null pointer");
  if (!workspace) return fail(VSG_ENOMEM, "workspace is NULL");
  DeviceGuard dg(pack->device);
  if (!dg.ok) return fail(VSG_ECUDA, "cannot select device %d", pack->device);
  cudaStream_t st = (cudaStream_t)stream;
  const int C = pack->cfg.flow_channels;
  Workspace ws(workspace, workspace_bytes);
  float* z = ws.take<float>((size_t)B * C * T);
  if (ws.overflow) return fail(VSG_ENOMEM, "workspace too small");
  const size_t mark = ws.off;
  int launches = 0;
  // z_p = (mu_p + noise * exp(logs_p)) * mask                       models/visinger.py:107
  // (tensor-core modes: drawn by the flow's first kernel while it lays the state out channels-last)
  const bool fuse_ps = precision != VSG_PRECISION_FP32 &&
                       (precision == VSG_PRECISION_BF16 || (x3_flow_on_tensor_cores() && !pack->flow_layers.empty() &&
                                                            pack->flow_layers[0].pre_x6[0].has_tmap));
  if (!fuse_ps) VSG_TRY(prior_sample(mu_p, logs_p, noise, mask, z, B, C, T, st));
  // z_q = flow(z_p, mask, g, reverse=True) * mask                    models/visinger.py:109
  // (tensor-core modes: the flow's last kernel writes z * mask straight into the caller's z_q buffer, which the decoder
  // then reads -- no separate mask pass, no copy)
  float* zq = z;
  bool masked = true;
  if (precision != VSG_PRECISION_FP32 && z_q_out) zq = z_q_out;
  bool sampled = false;
  VSG_TRY(run_flow(pack, fuse_ps ? mu_p : z, mask, g, zq, B, T, 1, precision, ws, st, &masked, fuse_ps ? logs_p : nullptr,
                   fuse_ps ? noise : nullptr, fuse_ps ? &sampled : nullptr));
  if (fuse_ps && !sampled) return fail(VSG_EINVAL, "internal: the flow did not draw the prior sample");
  if (!masked) VSG_TRY(mask_mul(zq, mask, zq, B, C, T, st));
  if (z_q_out && zq != z_q_out)
    VSG_CUDA_TRY(cudaMemcpyAsync(z_q_out, zq, (size_t)B * C * T * sizeof(float), cudaMemcpyDeviceToDevice, st));
  // wav = decoder(z_q * mask, g)                                      models/visinger.py:111
  ws.off = mark;   // the flow scratch is dead; the decoder reuses it
  if (precision == VSG_PRECISION_FP32) VSG_TRY(generator_forward_f32(pack, zq, g, wav, B, T, ws, st));
  else VSG_TRY(generator_forward_tc(pack, zq, g, wav, B, T, ws, st, precision == VSG_PRECISION_BF16X3));
  (void)launches;
  return VSG_OK;
}

extern "C" size_t vsg_posterior_workspace_bytes(const VsgPack* pack, int32_t B, int32_t T, int32_t precision) {
  if (check_common(pack, B, T, precision) != VSG_OK || !pack->has_enc) return 0;
  return (precision == VSG_PRECISION_BF16 ? posterior_ws_bytes_tc(pack, B, T) : posterior_ws_bytes_f32(pack, B, T)) + 1024;
}

extern "C" int vsg_posterior_forward(const VsgPack* pack, const float* x, const float* mask, const float* g,
                                     const float* noise, float* z_q, float* stats, int32_t B, int32_t T, int32_t precision,
                                     void* workspace, size_t workspace_bytes, void* stream) {
  reset_launch_counts();
  VSG_TRY(check_common(pack, B, T, precision));
  if (!pack->has_enc) return fail(VSG_EINVAL, "pack has no posterior encoder (create it with vsg_enc_pack_create)");
  if (B == 0 || T == 0) return VSG_OK;
  if (!x || !mask || !noise || !z_q || !stats) return fail(VSG_EINVAL, "null pointer");
  if (!workspace) return fail(VSG_ENOMEM, "workspace is NULL");
  DeviceGuard dg(pack->device);
  if (!dg.ok) return fail(VSG_ECUDA, "cannot select device %d", pack->device);
  Workspace ws(workspace, workspace_bytes);
  if (precision != VSG_PRECISION_BF16)
    return posterior_forward_f32(pack, x, mask, g, noise, z_q, stats, B, T, ws, (cudaStream_t)stream);
  return posterior_forward_tc(pack, x, mask, g, noise, z_q, stats, B, T, ws, (cudaStream_t)stream);
}

extern "C" size_t vsg_relenc_workspace_bytes(const VsgPack* pack, int32_t B, int32_t T, int32_t g_per_frame, int32_t precision) {
  if (check_common(pack, B, T, precision) != VSG_OK || !pack->has_relenc) return 0;
  return (precision == VSG_PRECISION_BF16 ? relenc_ws_bytes_tc(pack, B, T, g_per_frame) : relenc_ws_bytes_f32(pack, B, T, g_per_frame)) + 1024;
}

extern "C" int vsg_relenc_forward(const VsgPack* pack, const float* x, const float* mask, const float* g, int32_t g_per_frame,
                                  float* y, int32_t B, int32_t T, int32_t precision, void* workspace, size_t workspace_bytes,
                                  void* stream) {
  reset_launch_counts();
  VSG_TRY(check_common(pack, B, T, precision));
  if (!pack->has_relenc) return fail(VSG_EINVAL, "pack has no relative-position encoder (create it with vsg_relenc_pack_create)");
  if (B == 0 || T == 0) return VSG_OK;
  if (!x || !mask || !y) return fail(VSG_EINVAL, "null pointer");
  if (!workspace) return fail(VSG_ENOMEM, "workspace is NULL");
  DeviceGuard dg(pack->device);
  if (!dg.ok) return fail(VSG_ECUDA, "cannot select device %d", pack->device);
  Workspace ws(workspace, workspace_bytes);
  if (precision == VSG_PRECISION_BF16)
    return relenc_forward_tc(pack, x, mask, g, g_per_frame, y, B, T, ws, (cudaStream_t)stream);
  return relenc_forward_f32(pack, x, mask, g, g_per_frame, y, B, T, ws, (cudaStream_t)stream);
}

extern "C" size_t vsg_frame_prior_workspace_bytes(const VsgPack* pack, int32_t B, int32_t T, int32_t precision) {
  if (check_common(pack, B, T, precision) != VSG_OK || !pack->has_relenc || !pack->relenc.proj_w) return 0;
  return frame_prior_ws_bytes(pack, B, T, precision) + 1024;
}

extern "C" int vsg_frame_prior_forward(const VsgPack* pack, const float* x, const float* mask, const float* g,
                                       const float* noise, float* stats, float* z_p, int32_t B, int32_t T, int32_t precision,
                                       void* workspace, size_t workspace_bytes, void* stream) {
  reset_launch_counts();
  VSG_TRY(check_common(pack, B, T, precision));
  if (!pack->has_relenc || !pack->relenc.proj_w)
    return fail(VSG_EINVAL, "pack has no frame prior network (create it with vsg_frame_prior_pack_create)");
  if (B == 0 || T == 0) return VSG_OK;
  if (!x || !mask || !noise || !z_p) return fail(VSG_EINVAL, "null pointer");
  if (!workspace) return fail(VSG_ENOMEM, "workspace is NULL");
  DeviceGuard dg(pack->device);
  if (!dg.ok) return fail(VSG_ECUDA, "cannot select device %d", pack->device);
  Workspace ws(workspace, workspace_bytes);
  if (precision == VSG_PRECISION_BF16)
    return frame_prior_forward_tc(pack, x, mask, g, noise, stats, z_p, B, T, ws, (cudaStream_t)stream);
  return frame_prior_forward_f32(pack, x, mask, g, noise, stats, z_p, B, T, ws, (cudaStream_t)stream);
}

extern "C" int vsg_length_regulate(const float* enc, const int64_t* mel2ph, const float* pos_table, int32_t pos_rows,
                                   float* y, int32_t B, int32_t H, int32_t T_ph, int32_t T, void* stream) {
  reset_launch_counts();
  if (B < 0 || H <= 0 || T_ph < 0 || T < 0) return fail(VSG_EINVAL, "bad dimension");
  if (B == 0 || T == 0) return VSG_OK;
  if (!enc || !mel2ph || !y || (pos_table && pos_rows <= 0)) return fail(VSG_EINVAL, "null pointer");
  return length_regulate(enc, (const long long*)mel2ph, pos_table, pos_rows, y, B, H, T_ph, T, (cudaStream_t)stream);
}

extern "C" int vsg_infer_zp(const VsgPack* pack, const float* z_p, const float* mask, const float* g, float* wav,
                            float* z_q_out, int32_t B, int32_t T, int32_t precision, void* workspace, size_t workspace_bytes,
                            void* stream) {
  reset_launch_counts();
  VSG_TRY(check_common(pack, B, T, precision));
  if (!pack->has_flow || !pack->has_dec) return fail(VSG_EINVAL, "vsg_infer_zp needs a pack with both flow and decoder");
  if (pack->cfg.flow_channels != pack->cfg.dec_initial_channel)
    return fail(VSG_EINVAL, "flow channels (%d) != decoder initial_channel (%d)", pack->cfg.flow_channels,
                pack->cfg.dec_initial_channel);
  if (B == 0 || T == 0) return VSG_OK;
  if (!z_p || !mask || !wav) return fail(VSG_EINVAL, "null pointer");
  if (!workspace) return fail(VSG_ENOMEM, "workspace is NULL");
  DeviceGuard dg(pack->device);
  if (!dg.ok) return fail(VSG_ECUDA, "cannot select device %d", pack->device);
  Workspace ws(workspace, workspace_bytes);
  return infer_zp_run(pack, z_p, mask, g, wav, z_q_out, B, T, precision, ws, (cudaStream_t)stream);
}

namespace vsg {

int infer_zp_run(const VsgPack* pack, const float* z_p, const float* mask, const float* g, float* wav, float* z_q_out,
                 int B, int T, int precision, Workspace& ws, cudaStream_t st) {
  const int C = pack->cfg.flow_channels;
  float* z = ws.take<float>((size_t)B * C * T);
  if (ws.overflow) return fail(VSG_ENOMEM, "workspace too small");
  const size_t mark = ws.off;
  float* zq = z;                // (as in vsg_infer: the tensor-core flow writes z * mask straight into the caller's buffer)
  bool masked = true;
  if (precision != VSG_PRECISION_FP32 && z_q_out) zq = z_q_out;
  VSG_TRY(run_flow(pack, z_p, mask, g, zq, B, T, 1, precision, ws, st, &masked));
  if (!masked) VSG_TRY(mask_mul(zq, mask, zq, B, C, T, st));
  if (z_q_out && zq != z_q_out)
    VSG_CUDA_TRY(cudaMemcpyAsync(z_q_out, zq, (size_t)B * C * T * sizeof(float), cudaMemcpyDeviceToDevice, st));
  ws.off = mark;
  if (precision == VSG_PRECISION_FP32) VSG_TRY(generator_forward_f32(pack, zq, g, wav, B, T, ws, st));
  else VSG_TRY(generator_forward_tc(pack, zq, g, wav, B, T, ws, st, precision == VSG_PRECISION_BF16X3));
  return VSG_OK;
}

}  // namespace vsg

// ---- streaming windows ------------------------------------------------------------------------------------------------
// A window's frames [t0, t1) are computed exactly as the one-pass call computes them: the flow runs over
// [fa, fb) = [t0 - Cf - Cd, t1 + Cf + Cd) and the decoder over [da, db) = [t0 - Cd, t1 + Cd) of the flow's output (both
// clipped to [0, T), where the window's zero padding is the utterance's own), Cf / Cd being the receptive fields of the
// flow (reverse) and of the decoder in frames.  Each output is a function of the inputs in its receptive field only, every
// kernel sums each output in an order that does not depend on where the output sits in a tile (DESIGN.md 4.8), and the
// kernel choices are those of the whole batch (dec_window_needs_tc), so the central frames come out bit for bit.
namespace {

long long floor_div(long long a, long long b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }

}  // namespace

namespace vsg {

int wavenet_context(int kernel, int dilation_rate, int n_layers) {
  int r = 0, dil = 1;
  for (int i = 0; i < n_layers; ++i) {   // WaveNet in_layers: padding (K * dil - dil) / 2; pre / post are 1x1
    const int span = (kernel - 1) * dil, pad = (kernel * dil - dil) / 2;
    r += std::max(pad, span - pad);
    dil *= dilation_rate;
  }
  return r;
}

int flow_context(const VsgPack* p) {
  if (!p->has_flow) return 0;
  const VsgConfig& c = p->cfg;
  // each coupling layer widens the field by its WaveNet's reach
  return wavenet_context(c.flow_kernel_size, c.flow_dilation_rate, c.flow_n_layers) * c.flow_n_flows;
}

// Walk the receptive field of output frame 0 (samples [0, hop)) back through the decoder's layers, noting at every rate
// the frames its samples lie in: a window's tensor at that rate covers whole frames [da, db) of it.
int dec_context(const VsgPack* p) {
  if (!p->has_dec) return 0;
  const VsgConfig& c = p->cfg;
  long long R = p->hop, lo = 0, hi = p->hop - 1, left = 0, right = 0;
  auto note = [&]() { left = std::max(left, -floor_div(lo, R)); right = std::max(right, floor_div(hi, R)); };
  auto conv = [&](int k, int d) { const int pad = (k * d - d) / 2; lo -= pad; hi += (k - 1) * d - pad; };
  conv(p->conv_post_k, 1);   // conv_post, padding 3                     decoder.py:31,55-57
  note();
  for (int i = c.dec_n_ups - 1; i >= 0; --i) {
    long long rlo = 0, rhi = 0;   // the NK resblocks of a stage run in parallel on its upsampled input: the widest
    for (int j = 0; j < c.dec_n_kernels; ++j) {
      const long long lo0 = lo, hi0 = hi;
      const int k = c.dec_resblock_kernel_sizes[j];
      for (int q = c.dec_n_dilations[j] - 1; q >= 0; --q) {
        if (c.dec_resblock == 1) conv(k, 1);       // ResBlock1 conv2                      decoder.py:91-104
        conv(k, c.dec_resblock_dilations[j][q]);   // conv1 (ResBlock2: its only conv)     decoder.py:124-133
      }
      rlo = std::min(rlo, lo - lo0); rhi = std::max(rhi, hi - hi0);
      lo = lo0; hi = hi0;
    }
    lo += rlo; hi += rhi;
    note();
    // ups[i] = ConvTranspose1d(k, stride r, padding (k - r) / 2): y[n] = sum_m x[m] w[n + pad - m r]   decoder.py:24-26
    const int r = c.dec_upsample_rates[i], k = c.dec_upsample_kernel_sizes[i], pad = (k - r) / 2;
    lo = -floor_div(-(lo + pad - k + 1), r);
    hi = floor_div(hi + pad, r);
    R /= r;
    note();
  }
  conv(7, 1);   // conv_pre, padding 3                                    decoder.py:19
  note();
  return (int)std::max(left, right);
}

int window_needs(const VsgPack* p, int B, int T, int precision, int* need, int* align) {
  *need = 1; *align = 1;
  if (precision == VSG_PRECISION_FP32) return VSG_OK;   // the FFMA kernels choose nothing by length
  return dec_window_needs_tc(p, B, T, precision == VSG_PRECISION_BF16X3, need, align);
}

int window_ranges(const VsgPack* p, int B, int T, int t0, int t1, int precision, bool flow, WinRange* r, int Cp) {
  int need, A;
  VSG_TRY(window_needs(p, B, T, precision, &need, &A));
  const int Cd = dec_context(p), Cf = flow ? flow_context(p) : 0;
  int da = std::max(0, t0 - Cd) / A * A, db = std::min(T, (std::min(T, t1 + Cd) + A - 1) / A * A);
  if (db - da < need) {   // a kernel of the whole batch's choice needs a longer stage: widen, never switch kernels
    db = std::min(T, da + (need + A - 1) / A * A);
    if (db - da < need) da = std::max(0, (db - need) / A * A);
  }
  r->da = da; r->db = db;
  r->fa = std::max(0, da - Cf); r->fb = std::min(T, db + Cf);
  r->ga = std::max(0, da - 2 * Cf); r->gb = std::min(T, db + 2 * Cf);
  r->pa = std::max(0, da - 2 * Cf - Cp); r->pb = std::min(T, db + 2 * Cf + Cp);
  return VSG_OK;
}

int window_span(const VsgPack* p, int B, int T, int n, int precision) {
  if (check_common(p, B, T, precision) != VSG_OK || !p->has_dec || n < 1 || T < 1) return 0;
  int need, A;
  if (window_needs(p, B, T, precision, &need, &A) != VSG_OK) return 0;
  return std::min(T, std::max(std::min(n, T) + 2 * dec_context(p) + 2 * (A - 1), need + A - 1));
}

size_t window_ws(const VsgPack* p, int B, int T, int n, int precision) {
  const int Wd = window_span(p, B, T, n, precision);
  if (!Wd) return 0;
  const int Cf = flow_context(p), Wf = std::min(T, Wd + 2 * Cf);
  const size_t dec = precision == VSG_PRECISION_FP32 ? dec_ws_bytes_f32(p, B, Wd)
                                                     : dec_ws_bytes_tc(p, B, Wd, precision == VSG_PRECISION_BF16X3, T);
  const size_t z = p->has_flow ? align256((size_t)B * p->cfg.flow_channels * Wf * sizeof(float)) : 0;
  return z + std::max(flow_ws(p, B, Wf, precision), dec) + 1024;
}

// vsg_infer_zp_window after validation: z_p and mask hold frames [base, base + ld) of the batch in rows of ld frames
int zp_window_run(const VsgPack* pack, const float* z_p, const float* mask, int base, int ld, const float* g, float* wav,
                  int64_t wav_ld, float* z_q_out, int B, int T, int t0, int t1, int precision, Workspace& ws,
                  cudaStream_t st) {
  WinRange r;
  VSG_TRY(window_ranges(pack, B, T, t0, t1, precision, true, &r));
  const int C = pack->cfg.flow_channels, Tf = r.fb - r.fa;
  float* z = ws.take<float>((size_t)B * C * Tf);
  if (ws.overflow) return fail(VSG_ENOMEM, "workspace too small");
  const size_t mark = ws.off;
  // z_q = flow(z_p, mask, g, reverse=True) * mask over [fa, fb), read in place from the caller's rows
  bool masked = true;
  VSG_TRY(run_flow(pack, z_p + (r.fa - base), mask + (r.fa - base), g, z, B, Tf, 1, precision, ws, st, &masked, nullptr,
                   nullptr, nullptr, ld));
  if (!masked) VSG_TRY(mask_mul(z, mask + (r.fa - base), z, B, C, Tf, st, ld));
  if (z_q_out)
    VSG_CUDA_TRY(cudaMemcpy2DAsync(z_q_out, (size_t)(t1 - t0) * sizeof(float), z + (t0 - r.fa), (size_t)Tf * sizeof(float),
                                   (size_t)(t1 - t0) * sizeof(float), (size_t)B * C, cudaMemcpyDeviceToDevice, st));
  ws.off = mark;
  // wav = decoder(z_q) over [da, db); its samples of [t0, t1) straight into the caller's rows
  const DecWin w{T, Tf, (long long)wav_ld, (t0 - r.da) * pack->hop, (t1 - r.da) * pack->hop};
  const float* zd = z + (r.da - r.fa);
  if (precision == VSG_PRECISION_FP32) return generator_forward_f32(pack, zd, g, wav, B, r.db - r.da, ws, st, &w);
  return generator_forward_tc(pack, zd, g, wav, B, r.db - r.da, ws, st, precision == VSG_PRECISION_BF16X3, &w);
}

}  // namespace vsg

namespace {

int check_window(const VsgPack* pack, const void* in, float* wav, int64_t wav_ld, int B, int T, int t0, int t1,
                 int precision, void* workspace, size_t workspace_bytes) {
  VSG_TRY(check_common(pack, B, T, precision));
  if (!pack->has_dec) return fail(VSG_EINVAL, "pack has no decoder");
  if (t0 < 0 || t1 > T || t0 >= t1) return fail(VSG_EINVAL, "window [%d, %d) is not a non-empty part of [0, %d)", t0, t1, T);
  if (B == 0) return VSG_OK;
  if (!in || !wav) return fail(VSG_EINVAL, "null pointer");
  if (wav_ld < (int64_t)(t1 - t0) * pack->hop)
    return fail(VSG_EINVAL, "wav_ld %lld is shorter than the window's %lld samples", (long long)wav_ld,
                (long long)(t1 - t0) * pack->hop);
  if ((long long)T * pack->hop > 0x7fffffffLL / 4) return fail(VSG_EUNSUPPORTED, "sequence too long (%d frames)", T);
  if (!workspace) return fail(VSG_ENOMEM, "workspace is NULL");
  int need, A;
  VSG_TRY(window_needs(pack, B, T, precision, &need, &A));
  const size_t want = window_ws(pack, B, T, t1 - t0, precision);
  if (workspace_bytes < want) return fail(VSG_ENOMEM, "window workspace too small: need %zu bytes", want);
  return VSG_OK;
}

}  // namespace

extern "C" int vsg_window_context(const VsgPack* pack, int32_t* flow_frames, int32_t* dec_frames) {
  if (!pack || !flow_frames || !dec_frames) return fail(VSG_EINVAL, "null pointer");
  *flow_frames = flow_context(pack);
  *dec_frames = dec_context(pack);
  return VSG_OK;
}

extern "C" size_t vsg_window_workspace_bytes(const VsgPack* pack, int32_t B, int32_t T, int32_t max_frames,
                                             int32_t precision) {
  return window_ws(pack, B, T, max_frames, precision);
}

extern "C" int vsg_infer_zp_window(const VsgPack* pack, const float* z_p, const float* mask, const float* g, float* wav,
                                   int64_t wav_ld, float* z_q_out, int32_t B, int32_t T, int32_t t0, int32_t t1,
                                   int32_t precision, void* workspace, size_t workspace_bytes, void* stream) {
  reset_launch_counts();
  if (pack && (!pack->has_flow || !pack->has_dec))
    return fail(VSG_EINVAL, "vsg_infer_zp_window needs a pack with both flow and decoder");
  if (pack && pack->cfg.flow_channels != pack->cfg.dec_initial_channel)
    return fail(VSG_EINVAL, "flow channels (%d) != decoder initial_channel (%d)", pack->cfg.flow_channels,
                pack->cfg.dec_initial_channel);
  VSG_TRY(check_window(pack, z_p, wav, wav_ld, B, T, t0, t1, precision, workspace, workspace_bytes));
  if (B == 0) return VSG_OK;
  if (!mask) return fail(VSG_EINVAL, "null pointer");
  DeviceGuard dg(pack->device);
  if (!dg.ok) return fail(VSG_ECUDA, "cannot select device %d", pack->device);
  Workspace ws(workspace, workspace_bytes);
  return zp_window_run(pack, z_p, mask, 0, T, g, wav, wav_ld, z_q_out, B, T, t0, t1, precision, ws, (cudaStream_t)stream);
}

extern "C" int vsg_generator_forward_window(const VsgPack* pack, const float* z, const float* g, float* wav, int64_t wav_ld,
                                            int32_t B, int32_t T, int32_t t0, int32_t t1, int32_t precision,
                                            void* workspace, size_t workspace_bytes, void* stream) {
  reset_launch_counts();
  VSG_TRY(check_window(pack, z, wav, wav_ld, B, T, t0, t1, precision, workspace, workspace_bytes));
  if (B == 0) return VSG_OK;
  WinRange r;
  VSG_TRY(window_ranges(pack, B, T, t0, t1, precision, false, &r));
  DeviceGuard dg(pack->device);
  if (!dg.ok) return fail(VSG_ECUDA, "cannot select device %d", pack->device);
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(workspace, workspace_bytes);
  const DecWin w{T, T, (long long)wav_ld, (t0 - r.da) * pack->hop, (t1 - r.da) * pack->hop};
  if (precision == VSG_PRECISION_FP32) return generator_forward_f32(pack, z + r.da, g, wav, B, r.db - r.da, ws, st, &w);
  return generator_forward_tc(pack, z + r.da, g, wav, B, r.db - r.da, ws, st, precision == VSG_PRECISION_BF16X3, &w);
}
