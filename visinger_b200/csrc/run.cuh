// Internal declarations shared by the run drivers and the C-ABI entry points.
#pragma once
#include "vsg_common.cuh"

namespace vsg {

int launch_cond(const float* W, const float* bias, const float* g, float* out, int O, int I, int B, cudaStream_t st);
int prior_sample(const float* mu, const float* logs, const float* noise, const float* mask, float* z, int B, int C,
                 int T, cudaStream_t st);
int mask_mul(const float* x, const float* mask, float* y, int B, int C, int T, cudaStream_t st, int mask_ld = 0);

// The decoder over a window of frames of a longer batch (vsg_generator_forward_window / vsg_infer_zp_window): z holds the
// window's frames in rows of z_ld frames; wav row b (at wav + b * wav_ld) receives the window's samples [s0, s1).
// T_plan is the whole padded batch's length: every kernel choice that depends on a length is taken from it, so that a
// window computes each sample with the kernels -- and the rounding -- of the one-pass call.
struct DecWin {
  int T_plan;
  int z_ld;
  long long wav_ld;
  int s0, s1;
};

// output stage (output.cu): peak-normalise -> x 32767 -> int16 (utils/audio/io.py:8-14)
int wav_to_int16(const float* wav, const int32_t* lengths, int16_t* pcm, float* peak, int B, int L, int norm, cudaStream_t st);

// fp32 parity mode (run_f32.cu)
size_t flow_ws_bytes_f32(const VsgPack* P, int B, int T);
size_t dec_ws_bytes_f32(const VsgPack* P, int B, int T);
// x_ld > 0: x and mask are T frames of rows x_ld frames long (a window read in place); y is [B, C, T]
int flow_forward_f32(const VsgPack* P, const float* x, const float* mask, const float* g, float* y, int B, int T,
                     int reverse, Workspace& ws, cudaStream_t st, int x_ld = 0);
int generator_forward_f32(const VsgPack* P, const float* z, const float* g, float* wav, int B, int T, Workspace& ws,
                          cudaStream_t st, const DecWin* win = nullptr);

// bf16 tensor-core mode (run_tc.cu)
size_t flow_ws_bytes_tc(const VsgPack* P, int B, int T, int planes = 1);
// T_plan > 0: the decoder over T-frame windows of a T_plan-frame batch (sub-batch split taken from T_plan)
size_t dec_ws_bytes_tc(const VsgPack* P, int B, int T, bool x3, int T_plan = 0);
int flow_forward_tc(const VsgPack* P, const float* x, const float* mask, const float* g, float* y, int B, int T,
                    int reverse, Workspace& ws, cudaStream_t st, int planes = 1, const float* out_mask = nullptr,   // out_mask: y * mask
                    const float* ps_logs = nullptr, const float* ps_noise = nullptr,   // x = mu_p: prior sampling at the entry   // planes = 3: fp32 tolerance (bf16x3 mode)
                    int x_ld = 0);   // x_ld > 0: x and mask are T frames of rows x_ld frames long (a window read in place)
// VSG_X3_FLOW_FFMA=1 in the environment: the bf16x3 mode runs the flow on the fp32 CUDA-core kernels (A/B measurements)
bool x3_flow_on_tensor_cores();
int generator_forward_tc(const VsgPack* P, const float* z, const float* g, float* wav, int B, int T, Workspace& ws,
                         cudaStream_t st, bool x3, const DecWin* win = nullptr);
// What the kernels the one-pass decoder picks for a (B, T) batch ask of a window of it: at least *min_frames frames (the
// row-packed and fused kernels' shortest stage), starting and ending on multiples of *align frames (the row-packed
// kernels' time steps per row at each stage's rate).  VSG_EUNSUPPORTED if a chosen conv_post kernel has no window form.
int dec_window_needs_tc(const VsgPack* P, int B, int T, bool x3, int* min_frames, int* align);


// PosteriorEncoder (f32: run_f32.cu, bf16: run_tc.cu)
size_t posterior_ws_bytes_f32(const VsgPack* P, int B, int T);
size_t posterior_ws_bytes_tc(const VsgPack* P, int B, int T);
int posterior_forward_f32(const VsgPack* P, const float* x, const float* mask, const float* g, const float* noise,
                          float* z, float* stats, int B, int T, Workspace& ws, cudaStream_t st);
int posterior_forward_tc(const VsgPack* P, const float* x, const float* mask, const float* g, const float* noise,
                         float* z, float* stats, int B, int T, Workspace& ws, cudaStream_t st);


// y [B, Cout, T] = Conv1d(x [B, Cin, T]) with the fp32 kernel, stride 1, 'same' padding (run_f32.cu)
int conv_f32_plain(const ConvW32& w, const float* x, int B, int T, float* y, cudaStream_t st);

// RelativeEncoder (f32: run_f32.cu, bf16: run_tc.cu)
size_t relenc_ws_bytes_tc(const VsgPack* P, int B, int T, int g_t);
int relenc_forward_tc(const VsgPack* P, const float* x, const float* mask, const float* g, int g_t, float* y, int B, int T,
                      Workspace& ws, cudaStream_t st);
size_t relenc_ws_bytes_f32(const VsgPack* P, int B, int T, int g_t);
int relenc_forward_f32(const VsgPack* P, const float* x, const float* mask, const float* g, int g_t, float* y, int B, int T,
                       Workspace& ws, cudaStream_t st);


// FramePriorNetwork + prior sampling (encoder -> proj -> sample); stats [B, 2H, T] may be null
size_t frame_prior_ws_bytes(const VsgPack* P, int B, int T, int precision);
int frame_prior_forward_f32(const VsgPack* P, const float* x, const float* mask, const float* g, const float* noise,
                            float* stats, float* z, int B, int T, Workspace& ws, cudaStream_t st);
int frame_prior_forward_tc(const VsgPack* P, const float* x, const float* mask, const float* g, const float* noise,
                           float* stats, float* z, int B, int T, Workspace& ws, cudaStream_t st);
int length_regulate(const float* enc, const long long* mel2ph, const float* table, int table_rows, float* y, int B, int H,
                    int T_ph, int T, cudaStream_t st);

// vsg_flow_forward after validation (api.cu): the precision's flow kernels; see api.cu for masked / ps_* / sampled
int run_flow(const VsgPack* pack, const float* x, const float* mask, const float* g, float* y, int B, int T, int reverse,
             int precision, Workspace& ws, cudaStream_t st, bool* masked = nullptr, const float* ps_logs = nullptr,
             const float* ps_noise = nullptr, bool* sampled = nullptr, int x_ld = 0);

// The linear spectrogram (spec.cuh).  mask [B, T] = t < lengths[b] (lengths clamped to [0, T]).
// t0, T_len (a window): frames [t0, t0 + T) of a T_len-frame batch; T_len = 0 stands for T.
int lengths_mask(const int32_t* lengths, float* mask, int B, int T, cudaStream_t st, int t0 = 0, int T_len = 0);
size_t spec_frames_bytes(const SpecPack& S, int B, int T, bool tc);
// fp32: spec [B, bins, T] on the FFMA kernel (run_f32.cu)
int spectrogram_f32(const SpecPack& S, const float* wav, const int32_t* lengths, const float* mask, float* spec, int B,
                    int T, Workspace& ws, cudaStream_t st, int t0 = 0, int T_len = 0);
// bf16: u [B, T, in_pad] channels-last bf16 (the posterior's `pre` input, pad channels 0) on tcgen05 (run_tc.cu)
int spectrogram_tc(const VsgPack* P, const SpecPack& S, int in_pad, const float* wav, const int32_t* lengths,
                   const float* mask, __nv_bfloat16* u, int B, int T, Workspace& ws, cudaStream_t st, int t0 = 0,
                   int T_len = 0);
// [B, T, ld] bf16 -> [B, C, T] fp32
int widen_bf16(const __nv_bfloat16* x, float* y, int B, int C, int ld, int T, cudaStream_t st);
// the bf16 posterior from its channels-last input u [B, T, in_pad] (posterior_forward_tc after its transpose)
int posterior_core_tc(const VsgPack* P, const __nv_bfloat16* u, const float* mask, const float* g, const float* noise,
                      float* z, float* stats, int B, int T, Workspace& ws, cudaStream_t st);

// The per-launch test hooks' scope: a throw-away pack on `device` (weights, an error flag for the tensor-core kernels),
// freed on exit; finish() synchronises and reports a failed kernel (named `what`) or a set error flag.
struct DebugScope {
  VsgPack P;
  int* err = nullptr;
  int open(int device) {
    VSG_CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    VSG_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    P.device = device;
    P.sm_count = prop.multiProcessorCount;
    VSG_CUDA_TRY(cudaMalloc(&err, sizeof(int)));
    VSG_CUDA_TRY(cudaMemset(err, 0, sizeof(int)));
    return VSG_OK;
  }
  int finish(int rc, const char* what = "conv_tc_kernel") {
    if (rc != VSG_OK) return rc;
    cudaError_t ce = cudaDeviceSynchronize();
    if (ce != cudaSuccess) return fail(VSG_ECUDA, "%s execution failed: %s", what, cudaGetErrorString(ce));
    int h = 0;
    VSG_CUDA_TRY(cudaMemcpy(&h, err, sizeof(int), cudaMemcpyDeviceToHost));
    if (h) return fail(VSG_ECUDA, "%s set its error flag (%d)", what, h);
    return VSG_OK;
  }
  ~DebugScope() {
    if (err) cudaFree(err);
    for (void* q : P.allocs) cudaFree(q);
  }
};

// vsg_infer_zp after validation (api.cu): flow reverse from z_p, mask, decoder; shared with vsg_model_forward
int infer_zp_run(const VsgPack* pack, const float* z_p, const float* mask, const float* g, float* wav, float* z_q_out,
                 int B, int T, int precision, Workspace& ws, cudaStream_t st);

// ---- streaming windows (api.cu) ----
// Workspace of run_flow over T frames in `prec` (0 without a flow).
size_t flow_ws(const VsgPack* p, int B, int T, int prec);
// Receptive fields in latent frames each side (vsg_window_context): a WaveNet's (its in_layers' reach; pre / post 1x1),
// the flow's (one direction) and the decoder's.
int wavenet_context(int kernel, int dilation_rate, int n_layers);
int flow_context(const VsgPack* p);
int dec_context(const VsgPack* p);
// The ranges a window [t0, t1) of a (B, T) batch runs each part over, nested outward and clipped to [0, T): decoder
// [da, db) (widened and aligned for the whole batch's kernel choices), flow reverse [fa, fb) = +-Cf, flow forward
// [ga, gb) = +-2 Cf, spectrogram and posterior [pa, pb) = +-(2 Cf + Cp).
struct WinRange { int fa, fb, da, db, ga, gb, pa, pb; };
int window_ranges(const VsgPack* p, int B, int T, int t0, int t1, int precision, bool flow, WinRange* r, int Cp = 0);
// Upper bound of db - da over windows of up to n frames (0 on invalid arguments).
int window_span(const VsgPack* p, int B, int T, int n, int precision);
// Flow reverse + decoder scratch of windows of up to n frames (vsg_window_workspace_bytes; 0 on invalid arguments).
size_t window_ws(const VsgPack* p, int B, int T, int n, int precision);
// Frames [t0, t1) of vsg_infer_zp (vsg_infer_zp_window after validation): z_p and mask hold frames [base, base + ld) of
// the batch in rows of ld frames (the caller's [B, C, T] buffers: base 0, ld T).  Kernel choices come from (B, T).
int zp_window_run(const VsgPack* pack, const float* z_p, const float* mask, int base, int ld, const float* g, float* wav,
                  int64_t wav_ld, float* z_q_out, int B, int T, int t0, int t1, int precision, Workspace& ws,
                  cudaStream_t st);

}  // namespace vsg
