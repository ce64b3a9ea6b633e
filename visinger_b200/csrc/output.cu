// Output stage (SURVEY.md 8f, row f3): peak-normalise -> x 32767 -> int16, the arithmetic of the reference's
// `save_wav(norm=True)` (utils/audio/io.py:8-14; out_wav_norm: true, config/models/base_task.yaml:53) done on the
// device so that only int16 PCM crosses PCIe (half the bytes of the fp32 waveform).
//
// The reference does, in float32 numpy:  w = wav / np.abs(wav).max();  w = w * 32767;  w.astype(np.int16)
// i.e. one IEEE fp32 division, one IEEE fp32 multiplication and a conversion that truncates toward zero -- restated
// with __fdiv_rn / __fmul_rn / __float2int_rz so the integers are bit-identical.  The peak is taken over each
// utterance's VALID samples (the reference runs batch 1, tasks/visinger.py:246: a padded tail must not set the gain).
//
// HBM-bound glue: two passes over the waveform (4 B/sample read each) + 2 B/sample written.  Pass 1 is a per-utterance
// max-abs reduction (float4 loads, warp-shuffle + shared-memory tree, one atomicMax per block on the float bits --
// max is order-independent, so the result is run-to-run bit-stable); pass 2 scales and packs 8 samples per thread into
// one 16-byte store.
#include "vsg_common.cuh"
#include "run.cuh"

namespace vsg {

namespace {

constexpr int kPeakThreads = 256;

// grid (chunks, B); peak_bits[b] must be zeroed before the launch (non-negative floats order like their bit patterns)
__global__ void __launch_bounds__(kPeakThreads) wav_peak_kernel(const float* __restrict__ wav, const int32_t* __restrict__ lengths,
                                                                unsigned int* __restrict__ peak_bits, int L) {
  const int b = blockIdx.y;
  const int n = lengths ? min(max(lengths[b], 0), L) : L;
  const float* w = wav + (long long)b * L;
  float m = 0.f;
  const int n4 = ((reinterpret_cast<uintptr_t>(w) & 15) == 0) ? n / 4 : 0;     // rows of an odd L are not 16-byte aligned
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(w) + i);
    m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
  }
  for (int i = 4 * n4 + blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) m = fmaxf(m, fabsf(__ldg(w + i)));
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  __shared__ float sm[kPeakThreads / 32];
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x < 32) {
    m = threadIdx.x < kPeakThreads / 32 ? sm[threadIdx.x] : 0.f;
    for (int o = 4; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (threadIdx.x == 0 && m > 0.f) atomicMax(peak_bits + b, __float_as_uint(m));
  }
}

__device__ __forceinline__ int16_t to_pcm(float v, float peak, int norm) {
  if (norm) v = __fdiv_rn(v, peak);                     // wav / np.abs(wav).max()
  v = __fmul_rn(v, 32767.0f);                           // wav * 32767
  // numpy's float32 -> int16 cast goes through a 32-bit integer truncated toward zero and keeps its low 16 bits
  return (int16_t)__float2int_rz(v);
}

// 8 samples per thread; samples at or beyond an utterance's valid length are written as 0
__global__ void __launch_bounds__(256) wav_to_int16_kernel(const float* __restrict__ wav, const int32_t* __restrict__ lengths,
                                                           const unsigned int* __restrict__ peak_bits, int16_t* __restrict__ out,
                                                           int L, int norm) {
  const int b = blockIdx.y;
  const int n = lengths ? min(max(lengths[b], 0), L) : L;
  const float peak = __uint_as_float(peak_bits[b]);
  const float* w = wav + (long long)b * L;
  int16_t* o = out + (long long)b * L;
  const bool aligned = ((reinterpret_cast<uintptr_t>(w) & 15) == 0) && ((reinterpret_cast<uintptr_t>(o) & 15) == 0);
  for (int i0 = (blockIdx.x * blockDim.x + threadIdx.x) * 8; i0 < L; i0 += gridDim.x * blockDim.x * 8) {
    if (aligned && i0 + 8 <= n) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(w + i0)), c = __ldg(reinterpret_cast<const float4*>(w + i0) + 1);
      const float v[8] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
      uint32_t pk[4];
#pragma unroll
      for (int j = 0; j < 4; ++j)
        pk[j] = (uint32_t)(uint16_t)to_pcm(v[2 * j], peak, norm) | ((uint32_t)(uint16_t)to_pcm(v[2 * j + 1], peak, norm) << 16);
      *reinterpret_cast<uint4*>(o + i0) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    } else {
      for (int i = i0; i < min(i0 + 8, L); ++i) o[i] = i < n ? to_pcm(__ldg(w + i), peak, norm) : (int16_t)0;
    }
  }
}

}  // namespace

int wav_to_int16(const float* wav, const int32_t* lengths, int16_t* pcm, float* peak, int B, int L, int norm,
                 cudaStream_t st) {
  if ((long long)B * L == 0) return VSG_OK;
  unsigned int* peak_bits = reinterpret_cast<unsigned int*>(peak);
  VSG_CUDA_TRY(cudaMemsetAsync(peak_bits, 0, (size_t)B * sizeof(unsigned int), st));
  {
    const int per_block = kPeakThreads * 4 * 8;          // >= 8 float4 loads per thread
    dim3 grid((unsigned)std::max(1, std::min((L + per_block - 1) / per_block, 1184)), (unsigned)B);
    wav_peak_kernel<<<grid, kPeakThreads, 0, st>>>(wav, lengths, peak_bits, L);
    VSG_LAUNCH_CHECK("wav_peak_kernel");
  }
  {
    const int per_block = 256 * 8 * 2;
    dim3 grid((unsigned)std::max(1, std::min((L + per_block - 1) / per_block, 1184)), (unsigned)B);
    wav_to_int16_kernel<<<grid, 256, 0, st>>>(wav, lengths, peak_bits, pcm, L, norm);
    VSG_LAUNCH_CHECK("wav_to_int16_kernel");
  }
  return VSG_OK;
}

}  // namespace vsg

using namespace vsg;

extern "C" int vsg_wav_to_int16(const float* wav, const int32_t* lengths, int16_t* pcm, float* peak, int32_t B, int32_t L,
                                int32_t norm, void* stream) {
  reset_launch_counts();
  if (B < 0 || L < 0) return fail(VSG_EINVAL, "negative batch (%d) or length (%d)", B, L);
  if (B > 65535) return fail(VSG_EUNSUPPORTED, "batch %d exceeds 65535", B);
  if ((long long)B * L == 0) return VSG_OK;
  if (!wav || !pcm || !peak) return fail(VSG_EINVAL, "null pointer");
  return wav_to_int16(wav, lengths, pcm, peak, B, L, norm ? 1 : 0, (cudaStream_t)stream);
}
