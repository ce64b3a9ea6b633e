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

}  // namespace

namespace vsg {

// fp32: CUDA-core FFMA kernels.  bf16: tcgen05, one bf16 plane.  bf16x3: tcgen05 on three bf16 planes per value (the
// flow's z <= 1e-5 needs all 24 mantissa bits of its state; the decoder's 1e-4 is met by two planes).
// *masked (optional): in = the caller wants y * mask; out = true if the flow's last kernel applied it (tensor-core modes:
// the mask rides on the final layout change), false if the caller still has to
int run_flow(const VsgPack* pack, const float* x, const float* mask, const float* g, float* y, int B, int T, int reverse,
             int precision, Workspace& ws, cudaStream_t st, bool* masked, const float* ps_logs, const float* ps_noise,
             bool* sampled) {
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
                           sampled ? ps_logs : nullptr, sampled ? ps_noise : nullptr);
  }
  return flow_forward_f32(pack, x, mask, g, y, B, T, reverse, ws, st);
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
