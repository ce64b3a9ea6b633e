/*
 * visinger_b200.h -- C ABI of the B200-native VISinger inference hot path.
 *
 * The reference (jisang93/VISinger) is pure Python/PyTorch and has NO FFI, plugin or
 * operator interface of its own: the drop-in boundary is its nn.Module surface
 * (SURVEY.md section 8b).  This header is the C boundary underneath our mirror of that
 * surface; each entry point names the reference interface it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary;
 *   - activations are the reference's own tensors: fp32, [B, C, T] contiguous
 *     (time fastest), resident on the pack's CUDA device; `mask` is [B, 1, T] in {0,1};
 *     `g` is the speaker condition [B, gin, 1] or NULL (modules/visinger/flow.py:33,
 *     modules/visinger/decoder.py:40);
 *   - weights enter as the reference's state-dict entries (HOST fp32 pointers, the
 *     names and shapes of SURVEY.md Appendix A, either `weight_g`+`weight_v` or a
 *     plain `weight` after remove_weight_norm); vsg_pack_create folds weight-norm and
 *     the Flip permutations, re-lays the weights out for the kernels and uploads them;
 *   - the caller owns every input, output and workspace buffer; the library allocates
 *     device memory only inside vsg_pack_create and frees it in vsg_pack_destroy.
 *     No call synchronises the host or allocates: all run calls are asynchronous on
 *     `stream` (a cudaStream_t passed as void*) and CUDA-graph capturable;
 *   - every function returns 0 on success or a negative VSG_E* code and never throws;
 *     vsg_last_error() returns a thread-local, human readable message for the last
 *     failing call;
 *   - a VsgPack is immutable after creation and may be shared by several streams of
 *     its device; calls that share one workspace must be stream-ordered.
 */
#ifndef VISINGER_B200_H_
#define VISINGER_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VSG_ABI_VERSION 1

enum {
  VSG_OK = 0,
  VSG_EINVAL = -1,   /* bad argument / shape / missing weight             */
  VSG_ECUDA = -2,    /* a CUDA runtime or driver call failed               */
  VSG_ENOMEM = -3,   /* workspace too small / allocation failed            */
  VSG_EUNSUPPORTED = -4 /* configuration outside what the kernels implement */
};

/* Arithmetic mode of a run call. */
enum {
  VSG_PRECISION_FP32 = 0, /* fp32 storage, fp32 FFMA accumulate: the parity mode
                             (waveform max-abs <= 1e-4, flow z <= 1e-5 vs the reference) */
  VSG_PRECISION_BF16 = 1, /* bf16 operands + storage, fp32 accumulate on tcgen05 tensor
                             cores (TMEM accumulators, TMA-fed): the throughput mode     */
  VSG_PRECISION_BF16X3 = 2 /* split-bf16 on the same tensor-core kernels, fp32-mode tolerances on tcgen05.  Decoder:
                             every activation and weight is a (hi, lo) bf16 pair (~16 mantissa bits), every
                             product three MMAs (hi*hi + hi*lo + lo*hi).  Flow (z <= 1e-5 on a state of magnitude ~5):
                             three planes (hi, mid, lo = the fp32 value exactly), six plane products per MMA product,
                             issued small-first because the tensor pipe's fp32 accumulation truncates            */
};

#define VSG_MAX_UPS 8
#define VSG_MAX_RESBLOCK_KERNELS 4
#define VSG_MAX_RESBLOCK_DILATIONS 4

/* Constructor arguments of the two reference modules.  A part with n_flows == 0 /
 * n_ups == 0 is absent from the pack. */
typedef struct VsgConfig {
  /* ResidualCouplingBlock(channels, hidden_channels, kernel_size, dilation_rate,
   * n_layers, n_flows, gin_channels)            modules/visinger/flow.py:16-31 */
  int32_t flow_channels;
  int32_t flow_hidden;
  int32_t flow_kernel_size;
  int32_t flow_dilation_rate;
  int32_t flow_n_layers;
  int32_t flow_n_flows;
  int32_t flow_gin;
  /* Generator(initial_channel, resblock, resblock_kernel_sizes, resblock_dilation_sizes,
   * upsample_rates, upsample_initial_channel, upsample_kernel_sizes, gin_channels)
   *                                             modules/visinger/decoder.py:14-38 */
  int32_t dec_initial_channel;
  int32_t dec_resblock;      /* 1 = ResBlock1, 2 = ResBlock2 */
  int32_t dec_n_kernels;     /* len(resblock_kernel_sizes) */
  int32_t dec_resblock_kernel_sizes[VSG_MAX_RESBLOCK_KERNELS];
  int32_t dec_n_dilations[VSG_MAX_RESBLOCK_KERNELS];
  int32_t dec_resblock_dilations[VSG_MAX_RESBLOCK_KERNELS][VSG_MAX_RESBLOCK_DILATIONS];
  int32_t dec_n_ups;         /* len(upsample_rates) */
  int32_t dec_upsample_rates[VSG_MAX_UPS];
  int32_t dec_upsample_kernel_sizes[VSG_MAX_UPS];
  int32_t dec_upsample_initial_channel;
  int32_t dec_gin;
} VsgConfig;

/* One state-dict entry (host memory, fp32, contiguous). */
typedef struct VsgTensor {
  const char* name;   /* e.g. "flow.flows.0.enc.in_layers.2.weight_v", "decoder.ups.0.bias" */
  const float* data;
  int32_t ndim;
  int64_t shape[4];
} VsgTensor;

typedef struct VsgPack VsgPack;

/* ABI version of the loaded library (== VSG_ABI_VERSION of the header it was built from). */
int vsg_abi_version(void);

/* Thread-local message of the last failing call ("" if none). */
const char* vsg_last_error(void);

/*
 * One-time weight pre-pack.  Replaces what the reference does implicitly on every
 * forward: the weight_norm pre-hook (torch.nn.utils.weight_norm at
 * modules/visinger/encoder.py:147,154,164 and modules/visinger/decoder.py:24-26,72-87)
 * and Flip (modules/visinger/flow.py:88-95, folded into channel permutations of
 * pre/post).  `weights` uses the key layout of the reference checkpoint
 * ["state_dict"]["model"] (utils/commons/ckpt_utils.py:37-56) restricted to the two
 * modules: flow weights under prefix `flow_prefix`, decoder weights under `dec_prefix`
 * (e.g. "flow." / "decoder.", or "" when packing a stand-alone module).
 */
int vsg_pack_create(const VsgConfig* cfg, const VsgTensor* weights, int32_t n_weights,
                    const char* flow_prefix, const char* dec_prefix, int32_t device, VsgPack** out);
void vsg_pack_destroy(VsgPack* pack);

/* Bytes of caller-provided scratch each run call needs for (B, T) in `precision`
 * (the max over the three run calls).  0 on invalid arguments. */
size_t vsg_workspace_bytes(const VsgPack* pack, int32_t B, int32_t T, int32_t precision);

/*
 * Prior sampling, models/visinger.py:107:
 *   z_p = (mu_p + noise * exp(logs_p)) * mask         all [B, C, T], mask [B, 1, T]
 * `noise` is injected by the caller (the reference draws torch.randn_like(mu_p)).
 */
int vsg_prior_sample(const float* mu_p, const float* logs_p, const float* noise, const float* mask,
                     float* z_p, int32_t B, int32_t C, int32_t T, void* stream);

/*
 * ResidualCouplingBlock.forward(x, x_mask, g, reverse)   modules/visinger/flow.py:33-40
 * (coupling layers flow.py:66-85, WaveNet modules/visinger/encoder.py:167-195 with
 * fused_add_tanh_sigmoid_multiply encoder.py:206-213).  x, y: [B, channels, T]; y may
 * alias x.  `g` NULL iff flow_gin == 0.  reverse != 0 is the inference direction.
 */
int vsg_flow_forward(const VsgPack* pack, const float* x, const float* mask, const float* g, float* y,
                     int32_t B, int32_t T, int32_t reverse, int32_t precision,
                     void* workspace, size_t workspace_bytes, void* stream);

/*
 * Generator.forward(x, g)                                 modules/visinger/decoder.py:40-59
 * z: [B, initial_channel, T] -> wav: [B, 1, T * prod(upsample_rates)].
 */
int vsg_generator_forward(const VsgPack* pack, const float* z, const float* g, float* wav,
                          int32_t B, int32_t T, int32_t precision,
                          void* workspace, size_t workspace_bytes, void* stream);

/*
 * The whole inference hot path, models/visinger.py:107-111:
 *   z_p = (mu_p + noise*exp(logs_p))*mask ; z_q = flow(z_p, mask, g, reverse=True)*mask ;
 *   wav = decoder(z_q*mask, g)
 * `z_q_out` (may be NULL) receives z_q [B, channels, T].
 */
int vsg_infer(const VsgPack* pack, const float* mu_p, const float* logs_p, const float* noise,
              const float* mask, const float* g, float* wav, float* z_q_out,
              int32_t B, int32_t T, int32_t precision,
              void* workspace, size_t workspace_bytes, void* stream);

/*
 * Output stage, `save_wav(wav, path, sr, norm)` up to the file write        utils/audio/io.py:8-14
 * (called with norm = out_wav_norm: true at inference/visinger.py:100, tasks/visinger.py:258):
 *   pcm = int16( (norm ? wav / max|wav| : wav) * 32767 )     fp32 arithmetic, conversion truncating toward zero
 * -- the integers numpy produces, bit for bit.  wav: device fp32 [B, L] (the Generator's output); `lengths` (device
 * int32 [B], valid SAMPLES per utterance, or NULL = L): the peak is taken over the valid samples of each utterance
 * only (the reference runs one utterance per call) and samples beyond them are written as 0; pcm: device int16 [B, L];
 * peak: device fp32 [B], receives max|wav| per utterance.  Asynchronous on `stream`, no allocation, capturable.
 */
int vsg_wav_to_int16(const float* wav, const int32_t* lengths, int16_t* pcm, float* peak, int32_t B, int32_t L,
                     int32_t norm, void* stream);

/*
 * PosteriorEncoder(in_channels, out_channels, hidden_channels, kernel_size, dilation_rate, n_layers, gin_channels)
 *                                                                         modules/visinger/encoder.py:76-101
 * (constructed at models/visinger.py:59-60 as (num_linear_bins, 192, 192, 5, 1, 16, gin); the training / voice-conversion
 * side of the model: SURVEY.md section 8 row f4).  It re-uses the WaveNet kernels of the flow.
 */
typedef struct VsgEncConfig {
  int32_t in_channels;
  int32_t out_channels;
  int32_t hidden_channels;
  int32_t kernel_size;
  int32_t dilation_rate;
  int32_t n_layers;
  int32_t gin_channels;
} VsgEncConfig;

/* Pre-pack of a PosteriorEncoder's state-dict entries (`prefix` + "pre.weight", "enc.in_layers.0.weight_v", ...,
 * "proj.bias"); the result is an ordinary VsgPack (vsg_pack_destroy frees it) that only vsg_posterior_* accept. */
int vsg_enc_pack_create(const VsgEncConfig* cfg, const VsgTensor* weights, int32_t n_weights, const char* prefix,
                        int32_t device, VsgPack** out);
size_t vsg_posterior_workspace_bytes(const VsgPack* pack, int32_t B, int32_t T, int32_t precision);

/*
 * PosteriorEncoder.forward(x, nonpadding, g)                              modules/visinger/encoder.py:92-98
 *   h = pre(x) * mask ; h = WaveNet(h, mask, g) ; stats = proj(h) * mask ; (mu_q, logs_q) = split(stats)
 *   z_q = (mu_q + noise * exp(logs_q)) * mask
 * x: [B, in_channels, T]; noise: [B, out_channels, T] (the reference draws torch.randn_like(mu_q));
 * stats: [B, 2 * out_channels, T] receives proj(h) * mask -- mu_q and logs_q are its two channel halves, the views
 * torch.split returns; z_q: [B, out_channels, T].  FP32: FFMA kernels (reference parity); BF16: tcgen05 kernels
 * (BF16X3 runs as FP32, like the flow).
 */
int vsg_posterior_forward(const VsgPack* pack, const float* x, const float* mask, const float* g, const float* noise,
                          float* z_q, float* stats, int32_t B, int32_t T, int32_t precision,
                          void* workspace, size_t workspace_bytes, void* stream);

/*
 * RelativeEncoder(hidden_channels, filter_channels, n_heads, n_layers, kernel_size, p_dropout, window_size, block_length,
 * pre_ln=False, gin_channels)                                             modules/rel_transformer.py:257-320
 * -- the frame-rate stacks of the prior network (PitchPredictor, modules/visinger/predictor.py:7-19; FramePriorNetwork,
 * modules/visinger/encoder.py:58-73; SURVEY.md section 8 row f1) and the phoneme-rate stack of the TextEncoder.  Post-LN
 * only (pre_ln = False, the reference's default and the only variant VISinger builds), block_length = None, eval mode.
 */
typedef struct VsgRelEncConfig {
  int32_t hidden_channels;
  int32_t filter_channels;
  int32_t n_heads;
  int32_t n_layers;
  int32_t kernel_size;     /* FFN conv_1 taps */
  int32_t window_size;     /* relative-position window (4) */
  int32_t gin_channels;    /* 0 = no pre_net */
} VsgRelEncConfig;

int vsg_relenc_pack_create(const VsgRelEncConfig* cfg, const VsgTensor* weights, int32_t n_weights, const char* prefix,
                           int32_t device, VsgPack** out);
size_t vsg_relenc_workspace_bytes(const VsgPack* pack, int32_t B, int32_t T, int32_t g_per_frame, int32_t precision);

/*
 * RelativeEncoder.forward(x, x_mask, g)                                    modules/rel_transformer.py:286-320
 * x, y: [B, hidden, T] (y may alias x); mask: [B, 1, T]; g: NULL, or the condition the reference feeds to pre_net:
 * [B, gin, 1] (g_per_frame == 0, e.g. the speaker embedding of the PitchPredictor) or [B, gin, T] (g_per_frame != 0,
 * e.g. the frame-level f0 of the FramePriorNetwork).  Attention: full T x T softmax per head with +-window relative-
 * position key / value embeddings, masked scores filled with -1e4 (:167), channel LayerNorm eps 1e-4.
 * VSG_PRECISION_BF16 takes head widths hidden / n_heads of 16, 32, 48, 64 and 96 and windows <= 7, and returns
 * VSG_EUNSUPPORTED otherwise; the fp32 mode also takes head width 128.  Both take any T.  Beyond T = 2048 the bf16
 * attention runs over key chunks of 2048 frames plus a combine, and the workspace grows by about
 * ceil(T / 2048) * B * T * hidden * 4 bytes (vsg_relenc_workspace_bytes includes it).
 */
int vsg_relenc_forward(const VsgPack* pack, const float* x, const float* mask, const float* g, int32_t g_per_frame,
                       float* y, int32_t B, int32_t T, int32_t precision, void* workspace, size_t workspace_bytes,
                       void* stream);

/*
 * FramePriorNetwork(hidden, filter, n_heads, n_layers, kernel_size, gin_channels = 1, p_dropout)
 *                                                                         modules/visinger/encoder.py:58-73
 * with prior sampling fused behind it (SURVEY.md section 8 row f2).  Weights: `prefix` + "encoder.*" (a RelativeEncoder)
 * and `prefix` + "proj.{weight,bias}".
 *   h = encoder(x, mask, g) ; stats = proj(h) * mask ; (mu_p, logs_p) = split(stats)        encoder.py:70-73
 *   z_p = (mu_p + noise * exp(logs_p)) * mask                                               models/visinger.py:107
 * x: [B, hidden, T]; g: [B, 1, T] frame-level condition (log-f0 of voiced frames) or NULL; noise, z_p: [B, hidden, T];
 * stats: [B, 2 * hidden, T] or NULL (mu_p / logs_p are its channel halves).  z_p is what vsg_infer_zp consumes.
 */
int vsg_frame_prior_pack_create(const VsgRelEncConfig* cfg, const VsgTensor* weights, int32_t n_weights, const char* prefix,
                                int32_t device, VsgPack** out);
size_t vsg_frame_prior_workspace_bytes(const VsgPack* pack, int32_t B, int32_t T, int32_t precision);
int vsg_frame_prior_forward(const VsgPack* pack, const float* x, const float* mask, const float* g, const float* noise,
                            float* stats, float* z_p, int32_t B, int32_t T, int32_t precision,
                            void* workspace, size_t workspace_bytes, void* stream);

/*
 * Length regulator + frame positions (SURVEY.md section 8 row f2), one kernel:
 *   y[b, :, t] = enc[b, :, mel2ph[b, t] - 1]  (0 where mel2ph == 0)       expand_states, models/commons/align_ops.py:22-26
 *   y[b, :, t] += pos_table[pos_t, :],  pos_t = running count of frames with y[b, 0, t] != 0 (0 on the others)
 *                                                    models/visinger.py:79-82, modules/rel_transformer.py:78-100
 * enc: [B, H, T_ph]; mel2ph: int64 [B, T]; pos_table: [pos_rows, H] sinusoidal table (row 0 zero) or NULL; y: [B, H, T].
 */
int vsg_length_regulate(const float* enc, const int64_t* mel2ph, const float* pos_table, int32_t pos_rows, float* y,
                        int32_t B, int32_t H, int32_t T_ph, int32_t T, void* stream);

/* vsg_infer from an already sampled z_p (models/visinger.py:109-111): z_q = flow(z_p, reverse) * mask; wav = decoder(z_q). */
int vsg_infer_zp(const VsgPack* pack, const float* z_p, const float* mask, const float* g, float* wav, float* z_q_out,
                 int32_t B, int32_t T, int32_t precision, void* workspace, size_t workspace_bytes, void* stream);

/*
 * Streaming synthesis: flow and decoder over a window of latent frames.  Only the prior network needs the whole
 * utterance; everything downstream of z_p is convolutional with a finite receptive field, so a caller can sample z_p once
 * and then produce the waveform window by window -- to start playback early, or to interleave long requests -- with a
 * workspace that does not grow with T.  Every window is BIT-IDENTICAL to the same frames of the one-pass call, in all
 * three precisions: the flow runs over the window plus Cf + Cd frames of context each side and the decoder over the
 * window plus Cd, the length-dependent kernel choices are those of the whole (B, T) batch, and only the central samples
 * are stored (DESIGN.md section 4.8).  Concatenated windows equal the one-pass waveform; windows may come in any order.
 */
/* Context frames each side that a window needs for exact results: the flow's (reverse) and the decoder's receptive
 * fields in latent frames, derived from the pack's config (0 for an absent part).  Host only. */
int vsg_window_context(const VsgPack* pack, int32_t* flow_frames, int32_t* dec_frames);
/* Workspace of the window calls for windows of up to max_frames output frames of a (B, T) batch; it does not grow with T
 * (the sub-batch split the whole batch uses may make it smaller).  0 on invalid arguments. */
size_t vsg_window_workspace_bytes(const VsgPack* pack, int32_t B, int32_t T, int32_t max_frames, int32_t precision);
/* Frames [t0, t1) of vsg_infer_zp(z_p [B, C, T], mask [B, 1, T], g) bit for bit.  wav: row b at wav + b * wav_ld receives
 * the samples [t0 * hop, t1 * hop) of utterance b; z_q_out: NULL or fp32 [B, C, t1 - t0].  z_p and mask are read in place.
 * VSG_EINVAL: t0 < 0, t1 > T, t0 >= t1, a null pointer, wav_ld < (t1 - t0) * hop; VSG_ENOMEM: a workspace smaller than
 * vsg_window_workspace_bytes(B, T, t1 - t0); both before any launch.  No allocation, no synchronisation: capturable. */
int vsg_infer_zp_window(const VsgPack* pack, const float* z_p, const float* mask, const float* g, float* wav,
                        int64_t wav_ld, float* z_q_out, int32_t B, int32_t T, int32_t t0, int32_t t1, int32_t precision,
                        void* workspace, size_t workspace_bytes, void* stream);
/* The decoder alone: samples [t0 * hop, t1 * hop) of vsg_generator_forward(z [B, C, T], g) bit for bit, with the rules of
 * vsg_infer_zp_window. */
int vsg_generator_forward_window(const VsgPack* pack, const float* z, const float* g, float* wav, int64_t wav_ld,
                                 int32_t B, int32_t T, int32_t t0, int32_t t1, int32_t precision,
                                 void* workspace, size_t workspace_bytes, void* stream);

/*
 * The whole model: VISinger.forward(infer=True) from note tokens to waveform in one call
 * (VISinger(ph_dict_size, pitch_size, dur_size, hparams), the fields below; window_size is RelativeEncoder's 4,
 * spk_embed_dim the 256 inputs of spk_embed_proj).  The speaker condition has hot.flow_gin (= hot.dec_gin) channels.
 * use_pos_embed adds the sinusoidal frame positions to the prior input (models/visinger.py:79-82); the text encoder's own
 * positional term (modules/visinger/encoder.py:50-53) is always on, as VISinger builds its TextEncoder with it.
 */
typedef struct VsgModelConfig {
  int32_t ph_dict_size, pitch_size, dur_size;
  int32_t hidden, filter, n_heads, ffn_kernel_size, window_size;   /* hidden_size, ffn_filter_channels, num_heads */
  int32_t enc_layers, pitch_predictor_layers, frame_prior_layers;
  int32_t use_pos_embed, use_pitch_embed, use_spk_id, use_spk_embed, num_spk, spk_embed_dim;
  VsgConfig hot;   /* flow + decoder, as vsg_pack_create takes it */
} VsgModelConfig;

/*
 * Pre-pack of a whole VISinger state dict: `weights` are the checkpoint's entries under `prefix` ("" or "model.").
 * Builds the existing pack types inside (text_encoder.text_encoder.*, pitch_predictor.pitch_predictor.*, frame_prior.*,
 * flow.* + decoder.*) and uploads the token-rate weights: the three embedding tables, text_encoder.linear,
 * spk_id_proj / spk_embed_proj, pitch_predictor.linear.  posterior_encoder.*, phoneme_predictor.* and *._float_tensor are
 * ignored.  A missing required entry returns VSG_EINVAL naming it.
 *   Optional entry `prefix` + "embed_positions.freq" ([hidden / 2] fp32): the frequencies of the sinusoidal position
 * table, exp(k * -(ln 10000 / (hidden/2 - 1))), as the framework that made the reference's table computed them
 * (SinusoidalPositionalEmbedding.get_embedding evaluates that exp in fp32 with torch's CPU exp, which is not correctly
 * rounded).  Without it they are the correctly rounded fp32 values; at hidden = 192 one of the 96 differs from torch's by
 * one ulp, which moves the table by up to 7.6e-6 at position 30 000 (1.2e-4 at hidden = 256).
 * The result is freed by vsg_pack_destroy and accepted only by vsg_model_*.
 */
int vsg_model_pack_create(const VsgModelConfig* cfg, const VsgTensor* weights, int32_t n_weights, const char* prefix,
                          int32_t device, VsgPack** out);
/* Bytes of workspace vsg_model_forward needs for (B, T_ph, T) in `precision`; 0 on invalid arguments. */
size_t vsg_model_workspace_bytes(const VsgPack* pack, int32_t B, int32_t T_ph, int32_t T, int32_t precision);

/*
 * VISinger.forward(text_tokens, pitch_tokens, dur_tokens, mel2ph, spk_embed, spk_id, f0, uv, infer=True)
 * -> wav [B, T * hop] (and f0_pred, z_q).  Device pointers unless noted:
 *   text_tokens, pitch_tokens, dur_tokens: int64 [B, T_ph], 0 = padding; mel2ph: int64 [B, T], 1-based, 0 = padding;
 *   spk_id: HOST int64 [B] iff use_spk_id (else NULL), each in [0, num_spk) -- it is checked before anything is launched,
 *     so it is read at call time: a CUDA graph captured from this call replays the ids of the capture;
 *   spk_embed: fp32 [B, spk_embed_dim] iff use_spk_embed (else NULL);
 *   f0, uv: fp32 [B, T] each, or both NULL = the pitch predictor's own (f0 = pred[..., 0], voiced = pred[..., 1] <= 0;
 *     given: voiced = uv == 0); both must be NULL without use_pitch_embed;
 *   noise: fp32 [B, hidden, T] prior noise, or NULL: drawn as vsg_normal_noise(seeds) -- seeds: uint64 [B], used iff
 *     noise is NULL;
 *   wav: fp32 [B, T * hop]; f0_pred: fp32 [B, T, 2] or NULL (NULL without use_pitch_embed); z_q_out: fp32 [B, hidden, T]
 *     or NULL.
 * Precision: the RelativeEncoder stacks and the frame-prior head run bf16 in VSG_PRECISION_BF16 and fp32 otherwise; the
 * flow and decoder run as in vsg_infer_zp.  The token-rate glue (embeddings, Linear(3H -> H), speaker condition, pitch
 * head) is fp32 on CUDA cores in every mode.  Token and mel2ph values are device data and are not checked: an id outside
 * its table reads a zero row, a mel2ph entry above T_ph a padding frame.  Argument errors return VSG_EINVAL, a workspace
 * smaller than vsg_model_workspace_bytes VSG_ENOMEM, both before any launch.  Any T and T_ph the stacks take are accepted.
 */
int vsg_model_forward(const VsgPack* pack, const int64_t* text_tokens, const int64_t* pitch_tokens,
                      const int64_t* dur_tokens, const int64_t* mel2ph, const int64_t* spk_id, const float* spk_embed,
                      const float* f0, const float* uv, const float* noise, const uint64_t* seeds, float* wav,
                      float* f0_pred, float* z_q_out, int32_t B, int32_t T_ph, int32_t T, int32_t precision,
                      void* workspace, size_t workspace_bytes, void* stream);

/*
 * Voice conversion (VITS SynthesizerTrn.voice_conversion on VISinger's modules), from a waveform or a linear spectrogram:
 *   spec  = linear_spectrogram(wav)                          [B, bins, T], bins = n_fft / 2 + 1
 *   z     = posterior_encoder(spec, mask, g_src, noise)      (modules/visinger/encoder.py:92-98)
 *   z_hat = flow(flow(z, mask, g_src), mask, g_tgt, reverse) * mask
 *   wav'  = decoder(z_hat * mask, g_tgt)                     g_* = speaker_embedding of the source / target speaker
 *
 * vsg_convert_pack_create builds what vsg_model_pack_create builds (vsg_model_forward accepts the result and computes the
 * same bits on it) plus the `prefix` + "posterior_encoder.*" pack -- PosteriorEncoder(bins, hidden, hidden, kernel, 1,
 * n_layers, gin), bins, kernel and n_layers read from the weights -- and the spectrogram's DFT basis.  n_fft =
 * 2 * (bins - 1); the hop is the decoder's, prod(upsample_rates), so spectrogram frames are latent frames; win_length
 * (1 .. n_fft) is the periodic Hann window's length, zero-padded centrally to n_fft as torch.stft pads it.  VSG_EINVAL on
 * a missing entry (named in the message), on win_length outside [1, n_fft] and on n_fft < hop.
 *
 * The linear spectrogram (VITS spectrogram_torch, per utterance): frame f covers samples [f*hop - p, f*hop - p + n_fft),
 * p = (n_fft - hop) / 2 (rounded down); samples outside utterance b's own [0, lengths[b] * hop) are reflected about its
 * ends as torch's 'reflect' padding does (no edge repeat, folded again while outside);
 * spec = sqrt(re^2 + im^2 + 1e-6) * mask.  When n_fft - hop is even this is spectrogram_torch of the utterance alone,
 * frame for frame.  It runs as Conv1d(hop -> 2 * bins, ceil(win_length / hop)) over the signal cut into rows of hop
 * samples, with the window-folded DFT basis (evaluated in double, rounded once to fp32) as weights: on tcgen05 in bf16
 * (operands rounded to bf16, fp32 accumulation) in VSG_PRECISION_BF16, on the FFMA kernel in fp32 otherwise.
 *
 * Common arguments (device pointers unless noted):
 *   wav: fp32 [B, T * hop]; utterance b is its first lengths[b] * hop samples;
 *   lengths: int32 [B], valid latent frames per utterance; device data, clamped to [0, T] and not checked otherwise;
 *     mask [b, t] = t < lengths[b].
 * vsg_convert_workspace_bytes covers vsg_spectrogram and vsg_model_convert (0 on invalid arguments).
 */
int vsg_convert_pack_create(const VsgModelConfig* cfg, const VsgTensor* weights, int32_t n_weights, const char* prefix,
                            int32_t win_length, int32_t device, VsgPack** out);
size_t vsg_convert_workspace_bytes(const VsgPack* pack, int32_t B, int32_t T, int32_t precision);

/* spec: fp32 [B, bins, T].  In VSG_PRECISION_BF16 it holds the bf16 values the posterior consumes, widened. */
int vsg_spectrogram(const VsgPack* pack, const float* wav, const int32_t* lengths, float* spec, int32_t B, int32_t T,
                    int32_t precision, void* workspace, size_t workspace_bytes, void* stream);

/*
 * Exactly one of wav (fp32 [B, T * hop]) and spec (fp32 [B, bins, T], e.g. the reference's forward(..., mel=...) input).
 *   src_spk_id, tgt_spk_id: HOST int64 [B] iff use_spk_id (else NULL), range-checked before any launch (a CUDA graph
 *     captured from this call replays the ids of the capture); src_spk_embed, tgt_spk_embed: fp32 [B, spk_embed_dim] iff
 *     use_spk_embed;
 *   noise: fp32 [B, hidden, T] posterior noise, or NULL: vsg_normal_noise(seeds) (uint64 [B], used iff noise is NULL);
 *   wav_out: fp32 [B, T * hop]; spec_out: fp32 [B, bins, T] or NULL, the spectrogram of wav (NULL when spec is given);
 *   z_out: fp32 [B, hidden, T] or NULL, receives z_hat.
 * Precision: the spectrogram and the posterior run bf16 in VSG_PRECISION_BF16 and fp32 otherwise (as
 * vsg_posterior_forward); the flow runs in both directions and the decoder runs as in vsg_infer_zp.  The result equals
 * vsg_spectrogram -> vsg_posterior_forward -> vsg_flow_forward(reverse = 0) -> vsg_infer_zp bit for bit.  Argument errors
 * return VSG_EINVAL, a workspace smaller than vsg_convert_workspace_bytes VSG_ENOMEM, both before any launch.  No
 * allocation, no synchronisation: capturable.
 */
int vsg_model_convert(const VsgPack* pack, const float* wav, const float* spec, const int32_t* lengths,
                      const int64_t* src_spk_id, const float* src_spk_embed, const int64_t* tgt_spk_id,
                      const float* tgt_spk_embed, const float* noise, const uint64_t* seeds, float* wav_out,
                      float* spec_out, float* z_out, int32_t B, int32_t T, int32_t precision, void* workspace,
                      size_t workspace_bytes, void* stream);

/*
 * Streaming voice conversion: frames [t0, t1) of vsg_model_convert(wav, spec = NULL, ...) BIT FOR BIT, with a workspace
 * that does not grow with T.  Voice conversion has no attention: the spectrogram, the posterior's WaveNet, the flow (both
 * directions) and the decoder all have finite receptive fields, so a window of output frames depends on a bounded
 * stretch of input audio only.  A recording of any length converts in bounded memory, and audio that is still arriving
 * converts with a fixed look-ahead.  The decoder runs over [da, db) = the window plus Cd frames each side (widened for
 * the whole batch's kernel choices as in vsg_infer_zp_window), the flow reverse over [da - Cf, db + Cf), the flow
 * forward over [da - 2 Cf, db + 2 Cf), the spectrogram and the posterior over [da - 2 Cf - Cp, db + 2 Cf + Cp), all
 * clipped to [0, T) (DESIGN.md section 4.9).  Windows may come in any order; no state is kept between them.
 */
/* Context frames each side of a voice-conversion window: the posterior encoder's, the flow's (each direction) and the
 * decoder's receptive fields in latent frames.  Host only. */
int vsg_convert_window_context(const VsgPack* pack, int32_t* post_frames, int32_t* flow_frames, int32_t* dec_frames);
/* Host only.  The input that window [t0, t1) of a (B, T) batch reads: samples [*s0, *s1) of each utterance's row of wav,
 * with *s1 widened to cover every frame whose mask the window uses.  The window's result does not depend on samples
 * outside that span, and is the same for every lengths[b] with lengths[b] * hop >= *s1.  A live caller can emit
 * frames [t0, t1) as soon as samples [0, *s1) have arrived. */
int vsg_convert_window_input(const VsgPack* pack, int32_t B, int32_t T, int32_t t0, int32_t t1, int32_t precision,
                             int64_t* s0, int64_t* s1);
/* Does not grow with T.  0 on invalid arguments. */
size_t vsg_convert_window_workspace_bytes(const VsgPack* pack, int32_t B, int32_t T, int32_t max_frames, int32_t precision);
/* Frames [t0, t1) of vsg_model_convert(wav, spec = NULL, ...) bit for bit: wav_out row b at wav_out + b * wav_ld receives
 * samples [t0 * hop, t1 * hop); z_out: NULL or fp32 [B, hidden, t1 - t0] (z_hat).  wav [B, T * hop], lengths, noise
 * [B, hidden, T] are read in place; seeds / speaker arguments as in vsg_model_convert.  Argument and workspace rules of
 * vsg_infer_zp_window (VSG_EINVAL / VSG_ENOMEM before any launch); no allocation, no synchronisation, capturable. */
int vsg_model_convert_window(const VsgPack* pack, const float* wav, const int32_t* lengths,
                             const int64_t* src_spk_id, const float* src_spk_embed, const int64_t* tgt_spk_id,
                             const float* tgt_spk_embed, const float* noise, const uint64_t* seeds, float* wav_out,
                             int64_t wav_ld, float* z_out, int32_t B, int32_t T, int32_t t0, int32_t t1,
                             int32_t precision, void* workspace, size_t workspace_bytes, void* stream);

/*
 * Seeded standard-normal noise, out: fp32 [B, C, T].  Element (b, c, t) is Box-Muller on one Philox4x32-10 draw with
 * key (lo32(seeds[b]), hi32(seeds[b])) and counter (t, c, 0, 0): with x0, x1 its first two words,
 *   u1 = (x0 + 1) / 2^32,  u2 = x1 / 2^32,  out = fp32( sqrt(-2 ln u1) * cos(2 pi u2) )   (evaluated in double)
 * -- so an utterance's noise depends on its seed only, not on B, its batch neighbours or the padded length.
 * seeds: device uint64 [B].  Asynchronous, no allocation, capturable.
 */
int vsg_normal_noise(const uint64_t* seeds, float* out, int32_t B, int32_t C, int32_t T, void* stream);

/*
 * The sinusoidal position table vsg_model_forward builds in its workspace (SinusoidalPositionalEmbedding.get_embedding,
 * padding_idx 0): out[p, k] = sin(a), out[p, half + k] = cos(a) with a = fp32(p) * freq[k] rounded to fp32 and sin / cos
 * evaluated in double, rounded to fp32; row 0 and an odd dim's last column are 0.  freq: device fp32 [dim / 2], or NULL
 * for the correctly rounded values (see vsg_model_pack_create).  out: device fp32 [rows, dim].  Asynchronous.
 */
int vsg_debug_position_table(const float* freq, int32_t rows, int32_t dim, float* out, void* stream);

/* Samples produced per latent frame (prod(upsample_rates)); 0 if the pack has no decoder. */
int32_t vsg_hop_size(const VsgPack* pack);   /* (a model pack: its decoder's) */

/* Number of kernels launched by the most recent run call on this thread (bench bookkeeping). */
int32_t vsg_last_launch_count(void);
/* Launches of the convolution kernel per epilogue image in that call: out[i] = launches of image i (EPI_SIG_* numbering,
 * see vsg_debug_conv_tc), 0 beyond the library's images.  VSG_EINVAL if out is NULL or n < 0. */
int vsg_last_launch_images(int32_t* out, int32_t n);

/*
 * Per-layer parity hook (tests and tuning only; it allocates and synchronises, unlike the run calls):
 * one Conv1d on the bf16 tcgen05 kernel with its fused epilogue -- the unit the reference dispatches as
 * nn.Conv1d -> F.conv1d followed by the residual add / leaky_relu (modules/visinger/decoder.py:91-104).
 *   x_bf16: device bf16 [B, L, Cin] channels-last; w: HOST fp32 [Cout][Cin][k]; bias: HOST fp32 [Cout] or NULL;
 *   add0/add1: device bf16 [B, L, Cout] or NULL;
 *   v = (conv1d(x, w, dilation, padding = (k-1)*dilation/2) + bias + add0 + add1) * scale
 *   out_f32 (device fp32 [B, L, Cout] or NULL) = v; out_raw_bf16 = bf16(v); out_act_bf16 = bf16(leaky_relu(v, 0.1)).
 *   flags bit 0: HALO mode (one activation box per channel chunk, taps through row-shifted UMMA descriptors);
 *   bit 1: keep the weights resident in shared memory; bit 2: split-bf16 (x, add0, add1, out_raw, out_act then
 *   carry two bf16 planes per row: [B, L, 2*C] = [hi | lo]); bit 3: add0 holds leaky_relu(r, 0.1) of the residual r and
 *   is inverted in the epilogue (r = a > 0 ? a : 10 a); bits 4..: cap on 128-row blocks per tile (0 = 4).
 */
int vsg_debug_conv1d_bf16(const void* x_bf16, const float* w, const float* bias, const void* add0_bf16,
                          const void* add1_bf16, float scale, float* out_f32, void* out_raw_bf16, void* out_act_bf16,
                          int32_t B, int32_t L, int32_t Cin, int32_t Cout, int32_t k, int32_t dilation, int32_t flags,
                          int32_t device);

/*
 * Per-launch hook of the convolution kernel (tests only; allocates and synchronises): one launch with every epilogue
 * field and output geometry the library's own calls use.  B utterances, Cin -> Cout channels, k taps at dilation dil;
 * row q < Lq of the output (time step n = q * out_stride + out_phase < Lout) reads input rows q + in_off0 + j * dil
 * (zero outside 0 .. Lin - 1):
 *   linear (mode 0):  v = ((acc + bias + bcond) + add0 + add1) * scale [* mask]
 *   gate (mode 1):    output channel c of Cout / 2 = tanh(v[2c]) * sigmoid(v[2c + 1]), v = acc + bias + bcond
 *   couple (mode 2):  m = (acc + bias) * mask; out = (add0 - m) * mask (couple_sign < 0) | m + add0 * mask (> 0)
 * planes: bf16 planes per weight and activation value -- 1 plain bf16; 2 split-bf16 (hi, lo; linear mode only); 3 (hi,
 * mid, lo).  A tensor with several planes holds them part_stride (x: x_part_stride) channels apart in rows of ld (x: x_ld)
 * channels; 0 = the tensor's own width (rows [hi | lo]).  Planar layouts put whole planes apart: ld = C, part_stride =
 * B * L * C.  add0_is_act: add0 holds leaky_relu(r, slope) of the residual r, inverted in the epilogue.  out_raw = v,
 * out_act = leaky_relu(v, slope), each split into planes; out_f32 = v in fp32 [B, Lout, Cout (gate: Cout / 2)].
 * epi_sigs as in the library's defaults (2): 0 runs the generic image only, 1 adds ACT / RES_ACT / LINEAR, 2 the
 * running-sum images.  *image_out = the EPI_SIG_* image launched (GENERIC 0, ACT 1, RES_ACT 2, LINEAR 3, X6 4, SUM0 5,
 * SUM1 6, FINAL 7, ACT_X3 9, RES_ACT_X3 10, SUM0_X3 11, SUM1_X3 12, FINAL_X3 13).
 * x, add0, add1, out_raw, out_act, mask ([B][Lout]) and bcond ([B][bcond_bs] from output channel 0) are device pointers;
 * w (fp32 [Cout][Cin][k]) and bias (fp32 [Cout]) live on the host.  Optional pointers may be NULL.
 */
typedef struct VsgDebugConv {
  const void* x;
  const float* w;
  const float* bias;
  const float* bcond;
  const float* mask;
  const void* add0;
  const void* add1;
  void* out_raw;
  void* out_act;
  float* out_f32;
  int32_t planes, mode, couple_sign, add0_is_act, bcond_bs;
  float scale, slope;
  int32_t B, Lin, Cin, Cout, k, dil, in_off0, Lq, out_stride, out_phase, Lout;
  int32_t x_ld, x_part_stride, ld, part_stride;
  int32_t epi_sigs;
} VsgDebugConv;
int vsg_debug_conv_tc(const VsgDebugConv* d, int32_t* image_out, int32_t device);

/*
 * The decoder's upsampler as the generator launches it (tests only; allocates and synchronises):
 *   y = conv_transpose1d(x, w, bias, stride = rate, padding = (k - rate) / 2)   (modules/visinger/decoder.py:46)
 * w: HOST fp32 [Cin][Cout][k]; bias: HOST fp32 [Cout].  x: device bf16 [B, Lin, Cin]; out_act = leaky_relu(y, 0.1) and
 * out_raw = y (or NULL): device bf16 [B, Lin * rate, Cout]; out_f32: device fp32 [B, Lin * rate, Cout] or NULL (the fp32
 * copy runs the generic image; without it the production image runs).  flags bit 0: merged form (one convolution
 * Cin -> rate * Cout) instead of one launch per polyphase; bit 1: two bf16 planes per value; bit 2: planar input (planes
 * B * Lin * Cin apart; otherwise rows [hi | lo]); bit 3: planar outputs (planes B * Lin * rate * Cout apart).  The merged
 * two-plane form needs planar outputs.  *image_out = the EPI_SIG_* image of the last launch.
 */
int vsg_debug_upsample_tc(const void* x_bf16, const float* w, const float* bias, int32_t Cin, int32_t Cout, int32_t rate,
                          int32_t k, int32_t B, int32_t Lin, void* out_act_bf16, void* out_raw_bf16, float* out_f32,
                          int32_t flags, int32_t* image_out, int32_t device);

/*
 * Per-layer parity hook for the fused ResBlock1 pair kernel (tests and tuning only; allocates and synchronises):
 *   v = (conv1d(leaky_relu(conv1d(xa, w1, dilation d1) + b1, 0.1), w2) + b2 + add0 + add1) * scale
 * -- one (c1, c2) step of ResBlock1.forward (modules/visinger/decoder.py:91-104) with xa = leaky_relu(x) and add0 = x.
 *   xa_bf16, add0, add1, out_raw, out_act: device bf16 [B, L, C] channels-last; w1, w2: HOST fp32 [C][C][k];
 *   b1, b2: HOST fp32 [C]; out_f32: device fp32 [B, L, C] or NULL.  C in {16, 32}.
 */
int vsg_debug_pair_bf16(const void* xa_bf16, const float* w1, const float* b1, const float* w2, const float* b2,
                        const void* add0_bf16, const void* add1_bf16, float scale, float* out_f32, void* out_raw_bf16,
                        void* out_act_bf16, int32_t B, int32_t L, int32_t C, int32_t k, int32_t d1, int32_t device);

/*
 * The fused ResBlock1 pair kernel in every form the decoder launches it (tests only; allocates and synchronises):
 *   v = (conv1d(leaky_relu(conv1d(xa, w1, dilation d1) + b1, 0.1), w2) + b2 + residual + add1) * scale
 * residual = add0 (add0_is_act = 0) or the residual r recovered from add0 = leaky_relu(r, 0.1) (add0_is_act = 1: the
 * decoder's single activated stream).  xa, add0, add1, out_raw (bf16(v)), out_act (leaky_relu(v)): device bf16 [B, L, C]
 * channels-last; out_f32: device fp32 [B, L, C]; w1, w2: HOST fp32 [C][C][k]; b1, b2: HOST fp32 [C].  add0, add1 and the
 * outputs may be NULL.  C in {16, 32}.  *image_out = the EPI_SIG_* epilogue image of conv2 (see vsg_debug_conv_tc): an
 * fp32 copy runs the generic image, otherwise the image the decoder would launch.
 */
typedef struct VsgDebugPair {
  const void* xa;
  const float* w1;
  const float* b1;
  const float* w2;
  const float* b2;
  const void* add0;
  const void* add1;
  void* out_raw;
  void* out_act;
  float* out_f32;
  int32_t add0_is_act;
  float scale;
  int32_t B, L, C, k, d1;
} VsgDebugPair;
int vsg_debug_pair_tc(const VsgDebugPair* d, int32_t* image_out, int32_t device);

/*
 * Per-layer parity hook for the whole-ResBlock1 kernel (tests and tuning only; allocates and synchronises):
 *   for q in 0..n_pairs-1:  x = conv1d(leaky_relu(conv1d(leaky_relu(x), w[2q], dilation d_q) + b[2q]), w[2q+1]) + b[2q+1] + x
 *   out = (x [+ add1]) * scale
 * -- ResBlock1.forward (modules/visinger/decoder.py:91-104) in ONE kernel.  xa_bf16 = leaky_relu(x_0), add1, out_raw,
 * out_act: device bf16 [B, L, C] channels-last; w: HOST fp32 [2 * n_pairs][C][C][k]; b: HOST fp32 [2 * n_pairs][C];
 * dilations: HOST int32 [n_pairs]; out_f32: device fp32 [B, L, C] or NULL.  C in {16, 32, 64}.
 * max_mb caps the 128-row blocks per tile (0 = as many as fit), sets = epilogue warp sets (0 = default).
 */
int vsg_debug_resblock_bf16(const void* xa_bf16, const float* w, const float* b, int32_t n_pairs,
                            const int32_t* dilations, const void* add1_bf16, float scale, float* out_f32,
                            void* out_raw_bf16, void* out_act_bf16, int32_t B, int32_t L, int32_t C, int32_t k,
                            int32_t max_mb, int32_t sets, int32_t device);

/*
 * Per-kernel parity hooks of the relative-position encoder's attention (tests only; they synchronise):
 * MultiHeadAttention.attention (modules/rel_transformer.py:137-177, self-attention, heads_share = True) for n_heads heads
 * of width dk and relative-position window w:
 *   s_ij = (q_i . k_j + [|j-i| <= w] q_i . Ek[j-i+w]) / sqrt(dk);  s_ij = -1e4 where mask_i * mask_j == 0
 *   o_i = sum_j softmax_j(s)_ij (v_j + [|j-i| <= w] Ev[j-i+w])
 * mask: device fp32 [B, T]; ek, ev: device fp32 [2w+1][dk].
 *   _bf16: the tcgen05 kernel of the bf16 encoder.  qkv: device bf16 [B, T, 3 * n_heads * dk] channels-last (q | k | v,
 *   head h at channels h*dk ..); o: device bf16 [B, T, n_heads * dk].  dk in {16, 32, 48, 64, 96}, w <= 7, T <= 2048;
 *   VSG_EUNSUPPORTED otherwise (dk = 128 exceeds a B200 block's shared memory).  VSG_ECUDA if the kernel's error flag is set.
 *   _split_bf16: the split-key path of the bf16 encoder at any T: the same kernel over key chunks of key_chunk frames (a
 *   multiple of 128 up to 2048; 0 = 2048, what the encoder uses beyond T = 2048), then the combine of the chunks.  Same
 *   layouts, head widths and windows as _bf16; VSG_EINVAL for any other key_chunk.
 *   _f32: the fp32 kernel of the parity mode.  qkv: device fp32 [B, 3 * n_heads * dk, T]; o: device fp32 [B, n_heads * dk, T].
 */
int vsg_debug_attention_bf16(const void* qkv_bf16, const float* mask, const float* ek, const float* ev, void* o_bf16,
                             int32_t B, int32_t T, int32_t n_heads, int32_t dk, int32_t w, int32_t device);
int vsg_debug_attention_split_bf16(const void* qkv_bf16, const float* mask, const float* ek, const float* ev, void* o_bf16,
                                   int32_t B, int32_t T, int32_t n_heads, int32_t dk, int32_t w, int32_t key_chunk,
                                   int32_t device);
int vsg_debug_attention_f32(const float* qkv, const float* mask, const float* ek, const float* ev, float* o, int32_t B,
                            int32_t T, int32_t n_heads, int32_t dk, int32_t w, int32_t device);

/*
 * Per-kernel parity hook of the bf16 encoder's fused step after each residual add (tests only; synchronises), in place on
 * x (device bf16 [B, T, C] channels-last, C even and <= 256):
 *   x = (LayerNorm_C(x; gamma, beta, eps) [+ g]) * mask      (rel_transformer.py:24-42, :293-295)
 * gamma, beta: device fp32 [C]; g: device fp32 [B, C] (g_t = 0) or [B, C, T] (g_t = 1), or NULL; mask: device fp32 [B, T].
 */
int vsg_debug_layernorm_bf16(void* x_bf16, const float* gamma, const float* beta, const float* g, int32_t g_t,
                             const float* mask, float eps, int32_t B, int32_t T, int32_t C, int32_t device);

/*
 * Per-launch hooks of the fp32 (FFMA) mode's kernels (tests only; each allocates and synchronises, except the plan).
 * Argument errors return VSG_EINVAL before the device is touched.
 *
 * vsg_debug_conv_f32: one launch of the fp32 convolution kernel with every field the library's drivers set.  Layout
 * [B, C, T], time contiguous: element (b, c, t) of a tensor lives at b * *_bs + c * *_cs + t.  Output row q < Lq is time
 * step n = q * out_stride + out_phase (< Lout) and reads input steps q + in_off0 + j * dil (zero outside 0 .. Lin - 1),
 * through f(v) = leaky_relu(v, slope) if pre_lrelu (slope 0: ReLU), else v:
 *   v[co] = sum_{ci, j} w[co][ci][j] * f(x[b, ci, q + in_off0 + j * dil]) + bias[co] + bcond[b * bcond_bs + co]
 *   mk = mask[b * mask_bs + n] (1 without a mask)
 *   linear (epi 0):   u = (v + res[b, co, n]) * mk;  y[b, co, n] = u (acc_mode 0) | y + u (1) | (y + u) / acc_div (2)
 *   gate (epi 1):     y[b, c, n] = tanh(v[2c]) * sigmoid(v[2c + 1]) for c < Cout / 2
 *   res_skip (epi 2): co < rs_split: y[b, co, n] = (y + v) * mk;  otherwise y2[b, co - rs_split, n] = v (y2_first) or
 *                     y2 + v, times mk if y2_mask
 *   couple (epi 3):   m = v * mk; x1 = res[b, co, n] if res is given, else y[b, co, n];
 *                     y[b, co, n] = m + x1 * mk (couple_sign +1) | (x1 - m) * mk (couple_sign -1)
 *   magnitude (epi 4, VSG_DEBUG_F32_MAG; no bias or bcond): y[b, c, n] = sqrt(v[2c]^2 + v[2c + 1]^2 + 1e-6) * mk
 * (y + u in acc_mode 1 / 2 and the res_skip / couple forms read the old value at the same element.)  res may equal y.
 * gate_interleave (gate only): w and bias are the reference module's [tanh half | sigmoid half] order (channel c and c +
 * Cout / 2 form output c), packed by the library's interleave; bcond is then indexed in the packed order, channel c of
 * the tanh half at 2c and of the sigmoid half at 2c + 1.  Without it, w and bias are already in the packed order.
 * x, bcond, res, mask, y, y2: device fp32; w (fp32 [Cout][Cin][k]) and bias (fp32 [Cout] or NULL) live on the host.
 * tile_out[2] (or NULL) = { warps along the channels, warps along time } of the launched tile configuration.
 * VSG_EUNSUPPORTED (and no launch) where vsg_debug_conv_f32_plan refuses the shape.
 */
#define VSG_DEBUG_F32_MAG 4
typedef struct VsgDebugConvF32 {
  const float* x;
  const float* w;
  const float* bias;
  const float* bcond;
  const float* res;
  const float* mask;
  float* y;
  float* y2;
  int64_t x_bs, y_bs, res_bs, y2_bs;
  int32_t x_cs, y_cs, res_cs, y2_cs;
  int32_t B, Cin, Lin, Cout, k, dil, in_off0;
  int32_t pre_lrelu;
  float slope;
  int32_t bcond_bs, mask_bs;
  int32_t Lq, out_stride, out_phase, Lout;
  int32_t epi, acc_mode;
  float acc_div;
  int32_t rs_split, y2_first, y2_mask, couple_sign, gate_interleave;
} VsgDebugConvF32;
int vsg_debug_conv_f32(const VsgDebugConvF32* d, int32_t* tile_out, int32_t device);

/* Host only (no GPU): the tile plan of the fp32 convolution kernel for Cout output channels and k taps at dilation dil.
 * out[3] = { warps along the channels, warps along time, dynamic shared memory in bytes }: 2 x 4 warps (1024 time steps
 * per tile) for Cout <= 16, 4 x 2 (512) for Cout <= 32, else 8 x 1 (256); shared memory 4 * 8 * ((time steps per tile +
 * (k - 1) * dil) + k * channels per tile).  VSG_EUNSUPPORTED above 200 KB. */
int vsg_debug_conv_f32_plan(int32_t Cout, int32_t k, int32_t dil, int32_t* out);

/* The fp32 decoder's upsampler as the generator runs it: y = conv_transpose1d(leaky_relu(x, 0.1), w, bias, stride = rate,
 * padding = (k - rate) / 2) (modules/visinger/decoder.py:45-46) as `rate` polyphase launches of the fp32 convolution.
 * x: device fp32 [B, Cin, Lin]; y: device fp32 [B, Cout, Lin * rate]; w: HOST fp32 [Cin][Cout][k]; bias: HOST fp32 [Cout].
 * Needs k >= rate and k - rate even. */
int vsg_debug_upsample_f32(const float* x, const float* w, const float* bias, int32_t Cin, int32_t Cout, int32_t rate,
                           int32_t k, int32_t B, int32_t Lin, float* y, int32_t device);

/* The fp32 decoder's conv_post: wav = tanh(conv1d(leaky_relu(x, slope), w, padding = (k - 1) / 2)) (decoder.py:55-57), C
 * channels to one, no bias.  x: device fp32 [B, C, L]; w: HOST fp32 [C][k].  Samples n0 <= n < n1 of utterance b go to
 * wav[b * wav_ld + n - n0] (device fp32); nothing else is written.  Needs 0 <= n0 < n1 <= L and wav_ld >= n1 - n0. */
int vsg_debug_conv_post_f32(const float* x, const float* w, int32_t C, int32_t L, int32_t k, float slope, int32_t B,
                            int32_t n0, int32_t n1, float* wav, int64_t wav_ld, int32_t device);

/* The speaker-condition GEMV of every mode: out[b][o] = bias[o] + sum_i W[o][i] * g[b][i].  W [O][I], bias [O] (or NULL),
 * g [B][I], out [B][O]: device fp32. */
int vsg_debug_cond_f32(const float* W, const float* bias, const float* g, float* out, int32_t O, int32_t I, int32_t B,
                       int32_t device);

/* Tuning aids for tools/tune_plans.py: force the tile plan (0 / -1 = automatic) and the number of timed repetitions of
 * the following vsg_debug_conv1d_bf16 calls; average kernel milliseconds of the last such call. */
int vsg_debug_set_plan(int32_t mb, int32_t cw, int32_t two_ctas, int32_t resident, int32_t reps);
float vsg_debug_last_ms(void);

/* Host-only tuning aid: print (stderr) the tile plan the launcher would choose for one convolution.
 * x3: 0 plain bf16, 1 two bf16 planes per value (split-bf16), 2 three planes (the flow at the fp32 tolerance). */
int vsg_debug_plan(int32_t Cin, int32_t Cout, int32_t k, int32_t dilation, int32_t B, int32_t L, int32_t n_adds,
                   int32_t n_outs, int32_t x3);

/* Host-only (no GPU): the tile plan of the row-packed whole-ResBlock1 kernel for one resblock shape -- C channels, k taps,
 * n_pairs (conv1, conv2) pairs with the given dilations, L time steps per utterance.  variant: 0 plain bf16, 1 split-bf16
 * (bf16x3 mode), 2 plain bf16 as two CTAs per SM.  out[8] = { 128-row blocks per tile, halo time steps per side, valid
 * time steps per tile, weight-ring stages, dynamic shared memory in bytes, mask of the convolutions in the block-Toeplitz
 * form, tiles per utterance, tensor-memory columns }.  VSG_EUNSUPPORTED: the shape runs on the per-convolution kernels. */
int vsg_debug_rp_plan(int32_t C, int32_t k, int32_t n_pairs, const int32_t* dilations, int32_t L, int32_t variant,
                      int32_t* out);

/* Host-only (no GPU): the tile plan of the fused ResBlock1 pair kernel (see vsg_debug_pair_tc) for C channels, k taps,
 * conv1 dilation d1, L time steps per utterance, n_adds adds and n_outs bf16 outputs.  out[3] = { 128-row blocks per tile,
 * valid output rows per tile, tiles per utterance }.  VSG_EUNSUPPORTED: the decoder runs such a pair as two convolutions. */
int vsg_debug_pair_plan(int32_t C, int32_t k, int32_t d1, int32_t L, int32_t n_adds, int32_t n_outs, int32_t* out);

/* Process-wide tuning defaults of the tensor-core path: activation-operand feeding mode, resident weights, and the
 * L2-resident batch tiling of the decoder (target MB of one intermediate tensor per sub-batch, 0 = no tiling, <0 =
 * keep; minimum tiles per launch, <=0 = keep).
 * halo_mode is a bit field (A/B switches for bench.py and the tests; all off = the shipped configuration, halo_mode = 1):
 *   bit 0 HALO activation tiles | bit 1 bf16x3 mode without the row-packed resblock kernel | bit 2 row-packed kernel as
 *   two CTAs per SM (opt-in, measured equal) | bits 4-7 cap on 128-row blocks per tile | bit 8 no programmatic dependent launch |
 *   bit 9 no fused resblock pairs | bit 10 one launch per upsampler polyphase | bit 11 never split N = 256 tiles |
 *   bit 12 store raw AND activated resblock streams | bit 13 generic epilogue images only |
 *   bit 14 resblock chains of a stage on one stream | bit 15 whole-resblock kernel rb_tc (opt-in) | bits 16-20 cap on
 *   128-row blocks per resblock tile | bits 21-23 resblock epilogue warp sets (0 = 4) | bit 24 no row-packed resblock
 *   kernel | bit 25 row-packed kernel at C = 64 too | bit 26 no block-Toeplitz form | bit 27 no specialised images for
 *   the last conv2 of a resblock (running-sum epilogues) | bits 28-29 conv_post on the CUDA-core kernels (1 register
 *   window, 2 shared-memory window) instead of tcgen05 | bit 30 row-packed kernel with two epilogue warp sets per block |
 *   bit 31 flow with separate res / skip launches and one cond_layer GEMV per flow. */
int vsg_set_tc_options(int32_t halo_mode, int32_t w_resident, int32_t l2_tensor_mb, int32_t min_tiles);

#ifdef __cplusplus
}
#endif
#endif /* VISINGER_B200_H_ */
