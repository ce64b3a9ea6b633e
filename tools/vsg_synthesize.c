/*
 * vsg_synthesize: note tokens -> waveform through the C ABI alone (include/visinger_b200.h + libvisinger_b200.so).
 *
 *   gcc -O2 -std=c99 -Iinclude -I/usr/local/cuda/include tools/vsg_synthesize.c -Lvisinger_b200/lib -lvisinger_b200 \
 *       -L/usr/local/cuda/lib64 -lcudart -Wl,-rpath,visinger_b200/lib -o vsg_synthesize
 *   ./vsg_synthesize BUNDLE_DIR OUT.f32
 *
 * BUNDLE_DIR holds
 *   config.bin   the VsgModelConfig struct as raw bytes;
 *   weights.idx  one line per state-dict entry: "name ndim d0 .. d{ndim-1} offset" (offset in floats into weights.bin);
 *   weights.bin  raw float32;
 *   inputs.bin   raw int64: B, T_ph, T, precision, then text_tokens, pitch_tokens, dur_tokens [B, T_ph], mel2ph [B, T],
 *                spk_id [B] (speaker-id models), seeds [B].
 * OUT.f32 receives the waveform [B, T * hop] as raw float32.  Speaker-id models only (no spk_embed input).
 */
#define _POSIX_C_SOURCE 200809L   /* strdup */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <cuda_runtime_api.h>

#include "visinger_b200.h"

static void* read_file(const char* dir, const char* name, size_t* size) {
  char path[4096];
  snprintf(path, sizeof(path), "%s/%s", dir, name);
  FILE* f = fopen(path, "rb");
  if (!f) { fprintf(stderr, "cannot open %s\n", path); exit(1); }
  fseek(f, 0, SEEK_END);
  long n = ftell(f);
  fseek(f, 0, SEEK_SET);
  void* buf = malloc(n > 0 ? (size_t)n : 1);
  if (!buf || fread(buf, 1, (size_t)n, f) != (size_t)n) { fprintf(stderr, "cannot read %s\n", path); exit(1); }
  fclose(f);
  *size = (size_t)n;
  return buf;
}

#define CUDA_OK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { \
  fprintf(stderr, "%s: %s\n", #x, cudaGetErrorString(e_)); return 1; } } while (0)
#define VSG_OK_OR_DIE(x) do { int r_ = (x); if (r_ != VSG_OK) { \
  fprintf(stderr, "%s failed (%d): %s\n", #x, r_, vsg_last_error()); return 1; } } while (0)

/* device copy of n int64 values */
static int64_t* to_device(const int64_t* h, size_t n) {
  void* d = NULL;
  if (cudaMalloc(&d, n * sizeof(int64_t) + 1) != cudaSuccess) return NULL;
  if (cudaMemcpy(d, h, n * sizeof(int64_t), cudaMemcpyHostToDevice) != cudaSuccess) return NULL;
  return (int64_t*)d;
}

int main(int argc, char** argv) {
  if (argc != 3) { fprintf(stderr, "usage: %s BUNDLE_DIR OUT.f32\n", argv[0]); return 2; }
  const char* dir = argv[1];
  size_t n_cfg, n_blob, n_idx, n_in;
  VsgModelConfig* cfg = (VsgModelConfig*)read_file(dir, "config.bin", &n_cfg);
  if (n_cfg != sizeof(VsgModelConfig)) { fprintf(stderr, "config.bin: %zu bytes, expected %zu\n", n_cfg, sizeof(VsgModelConfig)); return 1; }
  if (cfg->use_spk_embed) { fprintf(stderr, "this tool feeds speaker ids only (use_spk_embed is set)\n"); return 1; }
  const float* blob = (const float*)read_file(dir, "weights.bin", &n_blob);
  char* idx = (char*)read_file(dir, "weights.idx", &n_idx);
  idx = (char*)realloc(idx, n_idx + 1);
  idx[n_idx] = 0;

  /* the weight table: one VsgTensor per index line, pointing into the blob */
  int cap = 1024, n_w = 0;
  VsgTensor* w = (VsgTensor*)calloc((size_t)cap, sizeof(VsgTensor));
  for (char* line = strtok(idx, "\n"); line; line = strtok(NULL, "\n")) {
    char name[512];
    int ndim, used = 0;
    if (sscanf(line, "%511s %d%n", name, &ndim, &used) != 2 || ndim < 0 || ndim > 4) { fprintf(stderr, "bad index line: %s\n", line); return 1; }
    if (n_w == cap) { cap *= 2; w = (VsgTensor*)realloc(w, (size_t)cap * sizeof(VsgTensor)); }
    VsgTensor* t = &w[n_w++];
    memset(t, 0, sizeof(*t));
    char* p = line + used;
    for (int d = 0; d < ndim; ++d) t->shape[d] = strtoll(p, &p, 10);
    long long off = strtoll(p, &p, 10);
    t->name = strdup(name);
    t->ndim = ndim;
    t->data = blob + off;
  }

  const int64_t* in = (const int64_t*)read_file(dir, "inputs.bin", &n_in);
  const int32_t B = (int32_t)in[0], T_ph = (int32_t)in[1], T = (int32_t)in[2], precision = (int32_t)in[3];
  const int64_t* text = in + 4;
  const int64_t* pitch = text + (size_t)B * T_ph;
  const int64_t* dur = pitch + (size_t)B * T_ph;
  const int64_t* mel2ph = dur + (size_t)B * T_ph;
  const int64_t* spk_id = cfg->use_spk_id ? mel2ph + (size_t)B * T : NULL;   /* host memory: range-checked by the call */
  const int64_t* seeds = mel2ph + (size_t)B * T + (cfg->use_spk_id ? B : 0);
  if (n_in != (size_t)(seeds + B - in) * sizeof(int64_t)) { fprintf(stderr, "inputs.bin has the wrong size\n"); return 1; }

  VsgPack* pack = NULL;
  VSG_OK_OR_DIE(vsg_model_pack_create(cfg, w, n_w, "", 0, &pack));
  const int32_t hop = vsg_hop_size(pack);
  const size_t ws_bytes = vsg_model_workspace_bytes(pack, B, T_ph, T, precision);
  const size_t n_wav = (size_t)B * T * hop;
  void *ws = NULL, *wav = NULL;
  CUDA_OK(cudaMalloc(&ws, ws_bytes));
  CUDA_OK(cudaMalloc(&wav, n_wav * sizeof(float)));
  int64_t *d_text = to_device(text, (size_t)B * T_ph), *d_pitch = to_device(pitch, (size_t)B * T_ph);
  int64_t *d_dur = to_device(dur, (size_t)B * T_ph), *d_mel2ph = to_device(mel2ph, (size_t)B * T);
  int64_t* d_seeds = to_device(seeds, (size_t)B);
  if (!d_text || !d_pitch || !d_dur || !d_mel2ph || !d_seeds) { fprintf(stderr, "device upload failed\n"); return 1; }

  VSG_OK_OR_DIE(vsg_model_forward(pack, d_text, d_pitch, d_dur, d_mel2ph, spk_id, NULL, NULL, NULL, NULL,
                                  (const uint64_t*)d_seeds, (float*)wav, NULL, NULL, B, T_ph, T, precision, ws, ws_bytes,
                                  NULL));
  float* h_wav = (float*)malloc(n_wav * sizeof(float));
  CUDA_OK(cudaMemcpy(h_wav, wav, n_wav * sizeof(float), cudaMemcpyDeviceToHost));
  FILE* f = fopen(argv[2], "wb");
  if (!f || fwrite(h_wav, sizeof(float), n_wav, f) != n_wav) { fprintf(stderr, "cannot write %s\n", argv[2]); return 1; }
  fclose(f);
  printf("synthesised B=%d x T=%d frames (T_ph=%d, hop %d, precision %d): %zu samples, %d kernel launches\n", B, T, T_ph,
         hop, precision, n_wav, vsg_last_launch_count());
  vsg_pack_destroy(pack);
  cudaFree(ws); cudaFree(wav);
  cudaFree(d_text); cudaFree(d_pitch); cudaFree(d_dur); cudaFree(d_mel2ph); cudaFree(d_seeds);
  return 0;
}
