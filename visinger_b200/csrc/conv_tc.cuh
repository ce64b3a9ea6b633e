// bf16 tensor-core implicit-GEMM convolution for sm_100a: tcgen05.mma with TMEM accumulators, operands
// staged in shared memory by TMA, warp-specialised and persistent.
//
// Activations are channels-last bf16 [B, L, C]; one CTA tile is 128 time steps (GEMM M = UMMA M = 128,
// one TMEM lane per time step) x N_TILE output channels (GEMM N <= 256) of one utterance.  The GEMM K
// dimension runs over (input-channel chunk, tap):
//     D[t, co] = sum_{chunk, tap} X[t + in_off0 + tap*dil, chunk] . W[tap][co, chunk]^T
//   * A operand: a [rows x KC] K-major box of X fetched by a 3-D TMA map (C, L, B).  Rows outside
//     [0, L) are zero-filled by the TMA unit -- that IS the convolution's zero padding and it also keeps
//     utterances of a batch apart.  In HALO mode one box of 128 + (ktaps-1)*dil rows is loaded per
//     channel chunk and every tap re-reads it through a row-shifted UMMA descriptor (A traffic / ktaps);
//     in RELOAD mode a fresh 128-row box is fetched per (chunk, tap).
//   * B operand: the pre-packed weights [tap][Cout][Cin] (K-major rows) through a 2-D TMA map.
//   * swizzle = KC*2 bytes (128B / 64B / 32B) on both operands, identical in the TMA map and the UMMA
//     shared-memory descriptor.
//   * small convolutions (all (chunk, tap) weight tiles <= ~100 KB) keep their weights RESIDENT in shared
//     memory for the whole persistent kernel: one TMA burst at start, no per-tap barrier round trips.
// ConvTranspose1d runs as `stride` polyphase launches of the same kernel (out_stride / out_phase).
//
// Warp roles (224 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer 0, warps 2..5 = epilogue,
// warp 6 = MMA issuer 1 (with mb >= 2 the two issuers take alternate 128-row blocks of the tile).  The producer and
// issuer warps run CONVERGED with `elect_one` around each TMA / tcgen05 instruction: that compiles to bare
// uniform-datapath instructions (UTCHMMA back to back), so the tensor pipe sets the pace -- 40 / 48 / 64 cycles per
// M=128 MMA at N <= 32 / 64 / 128 (tools/mma_bench2.cu) -- where a single-lane region cost ~80 cycles per instruction.
// A CTA tile is `mb` blocks of 128 time steps (mb = 1, 2 or 4) x N_TILE channels:
// every weight tile feeds mb MMAs (weight traffic / mb) and all per-tile costs (barrier waits, index math,
// TMA issue, staging synchronisation) are amortised over mb*128 rows -- the low-channel stages are bound by that
// overhead, not by HBM or tensor throughput.  The accumulator is double-buffered in TMEM (2 x mb x N_TILE
// columns) so the epilogue of tile i overlaps the main loop of tile i+1.
// Epilogue, per chunk of `cw` channels: each warp owns the rows of its TMEM lane quarter in every block:
// tcgen05.ld -> + bias (+ speaker condition) -> + residual / running resblock sum (one CTA-wide TMA load per
// chunk into swizzled shared memory, prefetched n_add_bufs-1 chunks ahead, across tiles) -> x scale / mask /
// gate / coupling -> raw value and leaky_relu(value) as bf16 into a CTA-wide swizzled staging tile
// [mb*128 rows x cw] -> ONE bulk TMA store per output.  All global traffic of the kernel is bulk TMA.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda.h>
#include <stdint.h>

namespace vsg {

constexpr int kMaxAChunks = 16;

struct ConvTC {
  int B, Lq, Lout;              // q positions per utterance, output length
  int KC, ktaps, dil, in_off0;
  // K loop: n_achunks activation chunks of KC channels at channel offset a_coff[c]; chunk c is multiplied with
  // n_wpass[c] weight column blocks at offsets w_coff[c][.] (plain bf16: one pass per chunk; split-bf16 "x3":
  // the hi chunk meets W_hi and W_lo, the lo chunk meets W_hi -- 3 MMAs per product, ~16 mantissa bits)
  int n_achunks;
  int a_coff[kMaxAChunks];
  int n_wpass[kMaxAChunks];
  int w_coff[kMaxAChunks][2];
  int n_wtiles;                 // sum of n_wpass * ktaps: weight tiles per n-tile
  int Cout, n_tile, n_ntiles, CoutT;   // CoutT: rows per tap in the packed weight matrix
  int n_parts, part_coff;       // epilogue tensors hold n_parts bf16 planes (hi[, lo]) part_coff channels apart
  int out_stride, out_phase;
  int mb;                       // 128-row blocks per tile
  int tile_stride;              // rows between consecutive tiles (128*mb, or less when a fused pair discards its halo rows)
  int m_tiles_per_b, total_tiles;
  int bar_slot0, tmem_col0;     // barrier bank / TMEM column offset of this half (fused pair: second conv uses bank 1)
  uint32_t a_off;               // start of the A ring inside shared memory (0 for the plain kernel)
  int t_row_off;                // fused pair: time of row 0 of the intermediate tile relative to the tile's first output row
  int halo_mode;                // 1: one A tile per channel chunk, taps via row-shifted descriptors
  int a_box_rows, a_n_boxes;    // the A tile is fetched as a_n_boxes TMA boxes of a_box_rows rows (<= 256 each)
  int w_resident;               // 1: all (chunk, tap) weight tiles are loaded once and stay in shared memory
  int stages_a, stages_w;
  uint32_t a_stage_bytes, w_stage_bytes, a_box_bytes, w_box_bytes;
  uint32_t w_off, e_off, bar_off;      // shared-memory carve-up, relative to the 1024-aligned base (A ring at 0)
  uint32_t tmem_cols;
  uint32_t swizzle_code;        // UMMA layout type: 2 = 128B, 4 = 64B, 6 = 32B
  uint32_t sbo_bytes;           // 8 rows * row bytes
  // epilogue: CTA-wide staging tiles of mb*128 rows x cw channels, moved by TMA in boxes of e_box_rows rows
  int cw, n_echunks;
  int e_box_rows, e_n_boxes;
  uint32_t e_buf_bytes, e_part_bytes, e_swz_mask;
  int n_add_bufs;
  // The epilogue runs on epi_sets (1 or 2) sets of 4 warps; with two sets (mb >= 2) set s takes the 128-row blocks
  // s, s + 2, ... of every tile.  A single set is one warp per SM sub-partition: latency-bound code with nothing to
  // overlap it with (ncu: the 4 warps busy ~80 % of the time, everything upstream waiting on them).  The sets share the
  // staging tiles, the add prefetch and the bulk stores (set 0's leader issues them); the named barriers span both.
  int epi_sets;
  int has_add0, has_add1;       // residual / running resblock sum: same geometry as the output, TMA-loaded
  int add0_is_act;              // add0 holds leaky_relu(x); the residual x is recovered as a > 0 ? a : a / slope.  In bf16
                                // that is as exact as storing x itself, and the producer then writes ONE tensor, not two
  int has_raw, has_act;         // outputs: value as is / leaky_relu(value), TMA-stored
  const float* bias;            // [Cout] or null
  const float* bcond; int bcond_bs;   // [B][bcond_bs] or null
  float scale;                  // applied after the adds
  float slope;                  // leaky_relu slope for out_act
  int mode;                     // EPI_TC_LINEAR / EPI_TC_GATE / EPI_TC_COUPLE
  const float* mask;            // [B][mask_ld] row mask or null (LINEAR: v *= mask; COUPLE: see below)
  int mask_ld;                  // floats between the mask rows of two utterances (Lout, or the whole batch's T for a window)
  int couple_sign;              // COUPLE: -1 reverse  x1 = (x1 - m) * mask,  +1 forward  x1 = m + x1 * mask
  uint32_t e_out_swz_mask;      // swizzle of the output staging rows (GATE halves the row width)
  float* out_f32;               // optional fp32 copy of the raw value [B, Lout, Cout] (debug / parity hook); EPI_TC_TANH: the output
  int tanh_cols;                // EPI_TC_TANH: out_f32[(b * Lq + q) * tanh_cols + i] = tanh(acc[i]), i < tanh_cols (<= 4)
  long long tanh_ld;            // EPI_TC_TANH, 0: as above; else only samples n = q * tanh_cols + i in [tanh_s0, tanh_s1) are
  int tanh_s0, tanh_s1;         //   stored, at out_f32[b * tanh_ld + n - tanh_s0] (a streaming window's central samples)
  int mag_ch;                   // EPI_TC_MAG: output channels >= mag_ch are written as 0 (the consumer's zero pad channels)
  int* error_flag;              // set to 1 if a barrier wait times out
};

enum : int { EPI_TC_LINEAR = 0, EPI_TC_GATE = 1, EPI_TC_COUPLE = 2, EPI_TC_TANH = 3, EPI_TC_MAG = 4 };

// Epilogue signatures: the decoder's two dominant epilogues get their own kernel instantiations in which every feature
// flag is a compile-time constant.  The generic kernel carries 12 epilogue variants (3 chunk widths x 4 modes; ~15 k SASS
// instructions, a quarter of a megabyte of code fetched by five different warp roles) and tests ~30 runtime flags per
// unit; a specialised one is a fifth of that.
//   EPI_SIG_GENERIC  everything decided at run time (flow, split-bf16, last conv of a resblock, debug hooks)
//   EPI_SIG_ACT      out_act = leaky_relu(acc + bias)                          (conv1 of a pair, merged upsamplers)
//   EPI_SIG_RES_ACT  out_act = leaky_relu(acc + bias + residual(add0_is_act))   (conv2 of a non-final pair)
//   EPI_SIG_LINEAR   plain-bf16 linear epilogue with run-time adds / outputs / scale but no speaker condition, mask or
//                    fp32 debug copy                                              (last conv2 of a resblock)
// (Separate images pay off for the decoder's long launches; the flow's ~20 us launches are better off sharing ONE warm
// image -- splitting the generic kernel per mode made the step slower.)
//   EPI_SIG_X6       the generic epilogue on THREE bf16 planes per tensor (hi, mid, lo = 24 mantissa bits: every fp32 value
//                    exactly), linear / gate / coupling with full-precision tanh / sigmoid: the flow at the fp32 tolerance
//   EPI_SIG_SUM0 / SUM1 / FINAL   the last conv2 of the stage's first / middle / last resblock: residual recovered from the
//                    activated stream, [+ running resblock sum,] -> raw running sum | x scale -> leaky_relu'd stage output
//                    (decoder.py:47-54).  On the run-time-flag image these launches cost 25 % more than a plain conv2.
enum : int { EPI_SIG_GENERIC = 0, EPI_SIG_ACT = 1, EPI_SIG_RES_ACT = 2, EPI_SIG_LINEAR = 3, EPI_SIG_X6 = 4,
             EPI_SIG_SUM0 = 5, EPI_SIG_SUM1 = 6, EPI_SIG_FINAL = 7,
             EPI_SIG_POST = 8,     // conv_post on the row-packed stage output: tanh of <= 4 accumulator columns -> fp32 waveform
             EPI_SIG_ACT_X3 = 9, EPI_SIG_RES_ACT_X3 = 10,   // ACT / RES_ACT on two bf16 planes per tensor (the bf16x3 decoder)
             EPI_SIG_SUM0_X3 = 11, EPI_SIG_SUM1_X3 = 12, EPI_SIG_FINAL_X3 = 13,
             EPI_SIG_MAG = 14,     // the linear spectrogram: |(re, im)| of interleaved channel pairs, masked, one bf16 output
             EPI_SIG_COUNT = 15 };

namespace tc {

__device__ __forceinline__ float tanh_fast(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must surface as an error, never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int* error_flag) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {
      if (error_flag) atomicExch(error_flag, 1);
      __trap();
    }
  }
}

__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
// TMA prefetch of one box into L2 (no shared-memory destination, no completion mechanism).
__device__ __forceinline__ void tma_prefetch_3d(const CUtensorMap* map, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// tcgen05.commit: arrive on `bar` once every MMA issued so far by this thread has completed.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// One lane of a CONVERGED warp.  `if (elect_one()) <tcgen05 instruction>` in warp-uniform control flow is the form the
// compiler turns into a bare uniform-datapath instruction; the same instruction inside an `if (lane == 0)` region is
// wrapped in a per-instruction ELECT / BRA.U.ANY loop with R2UR moves (~80 cycles per tcgen05.mma, measured).
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred = 0;
  asm volatile("{\n\t.reg .pred P1;\n\telect.sync _|P1, 0xffffffff;\n\tselp.u32 %0, 1, 0, P1;\n\t}" : "=r"(pred));
  return pred;
}

// D[tmem] (+)= A[smem] * B[smem]^T, bf16 inputs, fp32 accumulate, M = 128.
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// K-major shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
//   [0,14) start address >> 4 | [16,30) leading byte offset >> 4 (unused for swizzled K-major; 1)
//   [32,46) stride byte offset >> 4 (distance between 8-row groups) | [46,48) version = 1
//   [49,52) base offset | [61,64) layout type (2 = SWIZZLE_128B, 4 = 64B, 6 = 32B)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t sbo_bytes, uint32_t layout, uint32_t base_off) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1u << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1u << 46;
  d |= (uint64_t)(base_off & 7u) << 49;
  d |= (uint64_t)(layout & 7u) << 61;
  return d;
}

// Instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32 (bit 4), a/b format BF16 (bits 7, 10),
// both operands K-major, N >> 3 at [17,23), M >> 4 at [24,29).
__device__ __forceinline__ uint32_t make_idesc_bf16(uint32_t M, uint32_t N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// 16 consecutive fp32 accumulator columns of this thread's TMEM lane (no wait: pair with tmem_wait_ld).
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ void unpack_bf16x8(const uint4& u, float* f) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    f[2 * i] = __uint_as_float(w[i] << 16);
    f[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u);
  }
}

__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, const uint4& v) {
  asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
// TMA / UMMA swizzle: XOR the 16-byte-chunk index (address bits 4..6) with address bits 7..9 (masked by mode).
__device__ __forceinline__ uint32_t swz(uint32_t off, uint32_t mask) { return off ^ (((off >> 7) & mask) << 4); }

__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(src), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Walks this CTA's tiles (tile = blockIdx.x + i * gridDim.x) as (n-tile, m-tile, utterance) coordinates without
// per-tile integer divisions: the stride is decomposed once, then advanced with carries.
struct TileIter {
  int nt, mt, b, s_nt, s_mt, s_b, n_ntiles, m_tiles;
  __device__ __forceinline__ void init(int tile0, int step, int n_ntiles_, int m_tiles_) {
    n_ntiles = n_ntiles_; m_tiles = m_tiles_;
    nt = tile0 % n_ntiles; mt = (tile0 / n_ntiles) % m_tiles; b = tile0 / (n_ntiles * m_tiles);
    s_nt = step % n_ntiles; s_mt = (step / n_ntiles) % m_tiles; s_b = step / (n_ntiles * m_tiles);
  }
  __device__ __forceinline__ void next() {
    nt += s_nt;
    int c = nt >= n_ntiles ? 1 : 0;
    nt -= c ? n_ntiles : 0;
    mt += s_mt + c;
    c = mt >= m_tiles ? 1 : 0;
    mt -= c ? m_tiles : 0;
    b += s_b + c;
  }
};

constexpr int kThreads = 224;   // 7 warps: TMA producer, MMA issuer 0, 4 epilogue warps, MMA issuer 1
constexpr int kThreads2 = 352;  // + 4 warps: second epilogue set
constexpr int kMaxStages = 8;
constexpr int kMaxAddBufs = 4;
constexpr int kMaxCW = 64;
// barrier slots
constexpr int kBarAFull = 0, kBarAEmpty = kMaxStages, kBarWFull = 2 * kMaxStages, kBarWEmpty = 3 * kMaxStages;
constexpr int kBarAccFull = 4 * kMaxStages, kBarAccEmpty = kBarAccFull + 2, kBarAdd = kBarAccEmpty + 2;
constexpr int kNumBars = kBarAdd + kMaxAddBufs;
// named barriers of the 4 epilogue warps (id 0 is __syncthreads)
__device__ __forceinline__ void epi_bar_sync(int id, int n_threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n_threads) : "memory");
}

}  // namespace tc

// Plain-bf16 epilogue shortcuts on packed pairs (one HMUL2 + one HMNMX2 per TWO elements instead of two fp32
// instructions per element).  Both act on values that are already bf16, so they add one bf16 rounding of the scaled
// copy, which only matters for negative inputs; the split-bf16 (fp32-tolerance) mode does not use them.
__device__ __forceinline__ uint32_t bf16x2_scale_max(uint32_t a, float s) {   // max(a, a * s): leaky_relu for 0 < s < 1
  __nv_bfloat162 x = *reinterpret_cast<__nv_bfloat162*>(&a);
  __nv_bfloat162 y = __hmax2(x, __hmul2(x, __float2bfloat162_rn(s)));
  return *reinterpret_cast<uint32_t*>(&y);
}
__device__ __forceinline__ uint32_t bf16x2_scale_min(uint32_t a, float s) {   // min(a, a * s): inverse leaky_relu, s = 1 / slope > 1
  __nv_bfloat162 x = *reinterpret_cast<__nv_bfloat162*>(&a);
  __nv_bfloat162 y = __hmin2(x, __hmul2(x, __float2bfloat162_rn(s)));
  return *reinterpret_cast<uint32_t*>(&y);
}

// leaky_relu'd copy of OW fp32 values, plain bf16: pack, then max(r, r * slope) on the packed pairs.
template <int OW>
__device__ __forceinline__ void stage_out_act(const float* v, uint32_t base, uint32_t row_off, uint32_t swz_mask, float slope) {
  using namespace tc;
#pragma unroll
  for (int c = 0; c < OW / 8; ++c) {
    uint32_t h[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = bf16x2_scale_max(pack_bf16x2(v[8 * c + 2 * i], v[8 * c + 2 * i + 1]), slope);
    sts128(base + swz(row_off + c * 16, swz_mask), make_uint4(h[0], h[1], h[2], h[3]));
  }
}

// Write one row chunk of OW fp32 values into a swizzled bf16 staging tile: one plane (plain bf16), two planes
// hi = bf16(v), lo = bf16(v - hi) (split-bf16: the pair carries ~16 mantissa bits) or three (the fp32 value exactly).
template <int OW>
__device__ __forceinline__ void stage_out(const float* v, uint32_t base, uint32_t row_off, uint32_t swz_mask, int n_parts,
                                          uint32_t part_bytes) {
  using namespace tc;
#pragma unroll
  for (int c = 0; c < OW / 8; ++c) {
    uint32_t h[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = pack_bf16x2(v[8 * c + 2 * i], v[8 * c + 2 * i + 1]);
    const uint32_t addr = base + swz(row_off + c * 16, swz_mask);
    sts128(addr, make_uint4(h[0], h[1], h[2], h[3]));
    if (n_parts >= 2) {
      uint32_t l[4];
      float r0[4], r1[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        r0[i] = v[8 * c + 2 * i] - __uint_as_float(h[i] << 16);
        r1[i] = v[8 * c + 2 * i + 1] - __uint_as_float(h[i] & 0xFFFF0000u);
        l[i] = pack_bf16x2(r0[i], r1[i]);
      }
      sts128(addr + part_bytes, make_uint4(l[0], l[1], l[2], l[3]));
      if (n_parts == 3) {   // third plane: what the first two leave of the 24-bit mantissa (exact)
        uint32_t m[4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
          m[i] = pack_bf16x2(r0[i] - __uint_as_float(l[i] << 16), r1[i] - __uint_as_float(l[i] & 0xFFFF0000u));
        sts128(addr + 2u * part_bytes, make_uint4(m[0], m[1], m[2], m[3]));
      }
    }
  }
}

// MODE: EPI_TC_LINEAR  v = (acc + bias + bcond + add0 + add1) * scale [* mask]
//       EPI_TC_GATE    channel pairs (2c, 2c+1) hold the tanh / sigmoid halves (weights packed interleaved):
//                      out[c] = tanh(a) * sigmoid(s)  -- fused_add_tanh_sigmoid_multiply, encoder.py:206-213;
//                      the output tensor has Cout / 2 channels
//       EPI_TC_COUPLE  m = (acc + bias) * mask; out = (add0 - m) * mask | m + add0 * mask  (flow.py:78,83)
//       EPI_TC_TANH    wav = tanh(acc) of the first tanh_cols columns, fp32, straight to global memory (decoder.py:56-57)
//       EPI_TC_MAG     channel pairs (2c, 2c+1) hold (re, im) of one frequency bin (the window-folded DFT basis):
//                      out[c] = sqrt(re^2 + im^2 + 1e-6) * mask, 0 for c >= mag_ch; the output has Cout / 2 channels
template <int CW, int MODE, int NP, int SIG = EPI_SIG_GENERIC>
__device__ __forceinline__ void conv_tc_epilogue(const CUtensorMap& tmAdd0, const CUtensorMap& tmAdd1,
                                                 const CUtensorMap& tmRaw, const CUtensorMap& tmAct, const ConvTC& p,
                                                 uint32_t smem_base, uint32_t bar_base, uint32_t tmem_base, int warp,
                                                 int lane, int set = 0, int lead_warp = 2) {
  using namespace tc;
  bar_base += 8u * (uint32_t)p.bar_slot0;
  tmem_base += (uint32_t)p.tmem_col0;
  constexpr bool kPairs = MODE == EPI_TC_GATE || MODE == EPI_TC_MAG;   // two accumulator columns per output channel
  constexpr int OW = kPairs ? CW / 2 : CW;   // output channels per chunk
  const int tile_stride = p.tile_stride;
  const bool lead = (warp == lead_warp);   // this (converged) warp issues every epilogue TMA operation of the CTA
  const int n_sets = p.epi_sets > 1 ? 2 : 1;
  const int epi_threads = 128 * n_sets;
  const int quarter = warp & 3;          // tcgen05.ld: warp w may only touch TMEM lanes 32*(w%4) .. +31
  const int n_echunks = p.n_echunks, n_ntiles = p.n_ntiles, m_tiles_per_b = p.m_tiles_per_b, n_tile = p.n_tile;
  const int n_add_bufs = p.n_add_bufs, total_tiles = p.total_tiles, mb = p.mb;
  const int e_box_rows = p.e_box_rows, e_n_boxes = p.e_n_boxes;
  constexpr int n_parts = NP;            // bf16 planes per tensor: 1 = plain bf16, 2 = split-bf16 (hi, lo)
  const int part_coff = p.part_coff;
  const uint32_t e_buf_bytes = p.e_buf_bytes, swz_in = p.e_swz_mask, swz_out = p.e_out_swz_mask;
  const uint32_t part_bytes = p.e_part_bytes;     // one bf16 plane (hi or lo) of a staging buffer
  constexpr bool kGen = SIG == EPI_SIG_GENERIC || SIG == EPI_SIG_X6;
  constexpr bool kX3Sig = SIG == EPI_SIG_ACT_X3 || SIG == EPI_SIG_RES_ACT_X3 || SIG == EPI_SIG_SUM0_X3 || SIG == EPI_SIG_SUM1_X3 ||
                          SIG == EPI_SIG_FINAL_X3;
  constexpr bool kMag = SIG == EPI_SIG_MAG;
  static_assert(kGen || ((MODE == EPI_TC_LINEAR || (MODE == EPI_TC_TANH && SIG == EPI_SIG_POST) || (MODE == EPI_TC_MAG && kMag)) &&
                         NP == (kX3Sig ? 2 : 1)),
                "specialised signatures are linear epilogues on one bf16 plane (two for the _X3 images)");
  constexpr bool kRt = kGen || SIG == EPI_SIG_LINEAR;      // adds / outputs / scale decided at run time
  constexpr bool kSum0 = SIG == EPI_SIG_SUM0 || SIG == EPI_SIG_SUM0_X3, kSum1 = SIG == EPI_SIG_SUM1 || SIG == EPI_SIG_SUM1_X3,
                 kFinal = SIG == EPI_SIG_FINAL || SIG == EPI_SIG_FINAL_X3;
  constexpr bool kSum = kSum0 || kSum1 || kFinal;
  const bool has_add0 = kRt ? (p.has_add0 != 0) : (SIG == EPI_SIG_RES_ACT || SIG == EPI_SIG_RES_ACT_X3 || kSum);
  const bool has_add1 = kRt ? (p.has_add1 && MODE == EPI_TC_LINEAR) : (kSum1 || kFinal);
  const bool has_raw = kRt ? (p.has_raw != 0) : (kSum0 || kSum1 || kMag);
  const bool has_act = kRt ? (p.has_act && MODE == EPI_TC_LINEAR) : !(kSum0 || kSum1 || SIG == EPI_SIG_POST || kMag);
  const float scale = (kRt || kFinal) ? p.scale : 1.0f, slope = p.slope;
  const bool add0_is_act = kRt ? (p.add0_is_act != 0) : true;
  const float inv_slope = 1.0f / p.slope;
  const float* const bias = p.bias;
  const float* const bcond = kGen ? p.bcond : nullptr;
  const float* const maskp = (kGen || kMag) ? p.mask : nullptr;
  float* const out_f32 = kGen ? p.out_f32 : nullptr;
  int* const error_flag = p.error_flag;
  // staging carve-up: [add0 x n_add_bufs][add1 x n_add_bufs][raw x 2][act x 2], each e_buf_bytes
  const uint32_t add0_b = smem_base + p.e_off;
  const uint32_t add1_b = add0_b + (has_add0 ? (uint32_t)n_add_bufs * e_buf_bytes : 0u);
  const uint32_t raw_b = add1_b + ((kRt ? p.has_add1 != 0 : has_add1) ? (uint32_t)n_add_bufs * e_buf_bytes : 0u);
  const uint32_t act_b = raw_b + (has_raw ? 2u * e_buf_bytes : 0u);
  const bool has_add = has_add0 || has_add1;
  const bool has_out = has_raw || has_act;
  const uint32_t add_box_bytes = (uint32_t)e_box_rows * CW * 2u, out_box_bytes = (uint32_t)e_box_rows * OW * 2u;
  const uint32_t add_bytes = (uint32_t)((has_add0 ? 1 : 0) + (has_add1 ? 1 : 0)) * (uint32_t)(e_n_boxes * n_parts) * add_box_bytes;
  const uint32_t add_bar0 = bar_base + 8u * kBarAdd;
  const uint32_t acc_full0 = bar_base + 8u * kBarAccFull, acc_empty0 = bar_base + 8u * kBarAccEmpty;

  const int my_tiles = (total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  // add-operand prefetch cursor (leader only): walks (tile, chunk) units n_add_bufs-1 ahead of the consumers
  TileIter pf;
  pf.init((int)blockIdx.x, (int)gridDim.x, n_ntiles, m_tiles_per_b);
  int pf_cc = 0, pf_buf = 0, pf_left = my_tiles * n_echunks;
  auto issue_next_add = [&]() {
    if (pf_left <= 0) return;
    const int ch = pf.nt * n_tile + pf_cc * CW, row = pf.mt * tile_stride;
    const uint32_t bar = add_bar0 + 8u * pf_buf;
    if (elect_one()) {
      mbar_expect_tx(bar, add_bytes);
      for (int pt = 0; pt < n_parts; ++pt)
        for (int bx = 0; bx < e_n_boxes; ++bx) {
          const uint32_t off = pf_buf * e_buf_bytes + pt * part_bytes + bx * add_box_bytes;
          if (has_add0) tma_load_3d(add0_b + off, &tmAdd0, bar, ch + pt * part_coff, row + bx * e_box_rows, pf.b);
          if (has_add1) tma_load_3d(add1_b + off, &tmAdd1, bar, ch + pt * part_coff, row + bx * e_box_rows, pf.b);
        }
    }
    --pf_left;
    if (++pf_buf == n_add_bufs) pf_buf = 0;
    if (++pf_cc == n_echunks) { pf_cc = 0; pf.next(); }
  };
  if (has_add && lead) {
    for (int i = 0; i < n_add_bufs - 1; ++i) issue_next_add();
  }

  // bias is tile-invariant when the kernel has a single (n-tile, chunk): keep it in registers
  const bool bias_hoisted = (n_ntiles * n_echunks == 1) && bias != nullptr;
  float bias_r[CW];
#pragma unroll
  for (int i = 0; i < CW; ++i) bias_r[i] = 0.f;
  if (bias_hoisted) {
#pragma unroll
    for (int i = 0; i < CW; i += 4) {
      const float4 bv = __ldg(reinterpret_cast<const float4*>(bias + i));
      bias_r[i] = bv.x; bias_r[i + 1] = bv.y; bias_r[i + 2] = bv.z; bias_r[i + 3] = bv.w;
    }
  }

  int as = 0, add_buf = 0;
  uint32_t pacc = 0, add_phase = 0, out_count = 0;
  TileIter it;
  it.init((int)blockIdx.x, (int)gridDim.x, n_ntiles, m_tiles_per_b);
  for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, it.next()) {
    const int nt = it.nt, b = it.b;
    const int tile_row0 = it.mt * tile_stride;
    mbar_wait(acc_full0 + 8u * as, pacc, error_flag);
    fence_after_sync();
    const uint32_t taddr0 = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(as * mb * n_tile);
    for (int cc = 0; cc < n_echunks; ++cc) {
      if (has_add && lead) issue_next_add();     // refills the buffer drained by the previous unit (barrier B below)
      const int ch = nt * n_tile + cc * CW;
      const int och = kPairs ? ch / 2 : ch;
      if (has_add) {
        mbar_wait(add_bar0 + 8u * add_buf, (add_phase >> add_buf) & 1u, error_flag);
        add_phase ^= 1u << add_buf;
      }
      // staging buffer (out_count & 1) was last stored by the unit two back; barrier B of the previous unit already
      // published that store's read-completion (see below), so it can be overwritten without another barrier
      const uint32_t ob = (out_count & 1u) * e_buf_bytes;
      for (int bi = set; bi < mb; bi += n_sets) {
        const int srow = bi * 128 + quarter * 32 + lane;      // row inside the staging tile
        const int q = tile_row0 + srow;
        float v[CW];
        {
          uint32_t r[CW];
          const uint32_t taddr = taddr0 + (uint32_t)(bi * n_tile + cc * CW);
#pragma unroll
          for (int i = 0; i < CW / 16; ++i) tmem_ld16_nowait(taddr + (uint32_t)(i * 16), r + 16 * i);
          tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < CW; ++i) v[i] = __uint_as_float(r[i]);
        }
        if (cc == n_echunks - 1 && bi + n_sets >= mb) {   // accumulator drained: hand the TMEM stage back first
          fence_before_sync();
          __syncwarp();
          if (lane == 0) mbar_arrive(acc_empty0 + 8u * as);
        }
        float mk = 1.0f;
        if (maskp) mk = (q < p.Lq) ? __ldg(maskp + (long long)b * p.mask_ld + q) : 0.f;
        if (bias_hoisted) {
#pragma unroll
          for (int i = 0; i < CW; ++i) v[i] += bias_r[i];
        } else if (bias) {
#pragma unroll
          for (int i = 0; i < CW; i += 4) {
            const float4 bv = __ldg(reinterpret_cast<const float4*>(bias + ch + i));
            v[i] += bv.x; v[i + 1] += bv.y; v[i + 2] += bv.z; v[i + 3] += bv.w;
          }
        }
        if (bcond) {
          const float* bc = bcond + (long long)b * p.bcond_bs + ch;
#pragma unroll
          for (int i = 0; i < CW; i += 4) {
            const float4 bv = __ldg(reinterpret_cast<const float4*>(bc + i));
            v[i] += bv.x; v[i + 1] += bv.y; v[i + 2] += bv.z; v[i + 3] += bv.w;
          }
        }
        if (MODE == EPI_TC_COUPLE) {
#pragma unroll
          for (int i = 0; i < CW; ++i) v[i] *= mk;     // m = post(h) * mask
        }
        if (has_add) {
          const uint32_t row_off_in = (uint32_t)srow * (CW * 2);
          if (has_add0) {
            const uint32_t base = add0_b + add_buf * e_buf_bytes;
#pragma unroll
            for (int c = 0; c < CW / 8; ++c) {
              float f[8];
              uint4 u = lds128(base + swz(row_off_in + c * 16, swz_in));
              if (add0_is_act && n_parts == 1) {   // residual = a > 0 ? a : a / slope = min(a, a / slope), on packed pairs
                u.x = bf16x2_scale_min(u.x, inv_slope); u.y = bf16x2_scale_min(u.y, inv_slope);
                u.z = bf16x2_scale_min(u.z, inv_slope); u.w = bf16x2_scale_min(u.w, inv_slope);
              }
              unpack_bf16x8(u, f);
              if (n_parts >= 2) {
                float g2[8];
                unpack_bf16x8(lds128(base + part_bytes + swz(row_off_in + c * 16, swz_in)), g2);
#pragma unroll
                for (int i = 0; i < 8; ++i) f[i] += g2[i];
                if (n_parts == 3) {
                  unpack_bf16x8(lds128(base + 2u * part_bytes + swz(row_off_in + c * 16, swz_in)), g2);
#pragma unroll
                  for (int i = 0; i < 8; ++i) f[i] += g2[i];
                }
                if (add0_is_act) {   // split planes: the same recovery on the fp32 sum of the planes
#pragma unroll
                  for (int i = 0; i < 8; ++i) f[i] = fminf(f[i], f[i] * inv_slope);
                }
              }
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                if (MODE == EPI_TC_COUPLE) v[8 * c + i] = p.couple_sign < 0 ? (f[i] - v[8 * c + i]) * mk : v[8 * c + i] + f[i] * mk;
                else v[8 * c + i] += f[i];
              }
            }
          }
          if (has_add1) {
            const uint32_t base = add1_b + add_buf * e_buf_bytes;
#pragma unroll
            for (int c = 0; c < CW / 8; ++c) {
              float f[8];
              unpack_bf16x8(lds128(base + swz(row_off_in + c * 16, swz_in)), f);
              if (n_parts >= 2) {
                float g2[8];
                unpack_bf16x8(lds128(base + part_bytes + swz(row_off_in + c * 16, swz_in)), g2);
#pragma unroll
                for (int i = 0; i < 8; ++i) f[i] += g2[i];
                if (n_parts == 3) {
                  unpack_bf16x8(lds128(base + 2u * part_bytes + swz(row_off_in + c * 16, swz_in)), g2);
#pragma unroll
                  for (int i = 0; i < 8; ++i) f[i] += g2[i];
                }
              }
#pragma unroll
              for (int i = 0; i < 8; ++i) v[8 * c + i] += f[i];
            }
          }
        }
        if (MODE == EPI_TC_LINEAR) {
          if (scale != 1.0f) {
#pragma unroll
            for (int i = 0; i < CW; ++i) v[i] *= scale;
          }
          if (maskp) {
#pragma unroll
            for (int i = 0; i < CW; ++i) v[i] *= mk;
          }
        }
        if (MODE == EPI_TC_GATE) {
#pragma unroll
          for (int c = 0; c < CW / 2; ++c) {
            if (NP == 1) {
              const float t = tanh_fast(v[2 * c]);
              const float sg = 0.5f * tanh_fast(0.5f * v[2 * c + 1]) + 0.5f;   // sigmoid(x) = (1 + tanh(x/2)) / 2
              v[c] = t * sg;
            } else {   // fp32-tolerance modes: the libm-grade functions of the fp32 kernels (kernels_f32.cuh)
              v[c] = tanhf(v[2 * c]) * (1.0f / (1.0f + expf(-v[2 * c + 1])));
            }
          }
        }
        if (MODE == EPI_TC_MAG) {
#pragma unroll
          for (int c = 0; c < CW / 2; ++c)
            v[c] = och + c < p.mag_ch ? sqrtf(fmaf(v[2 * c], v[2 * c], fmaf(v[2 * c + 1], v[2 * c + 1], 1e-6f))) * mk : 0.f;
        }
        if (MODE == EPI_TC_TANH) {   // one 16-byte store per row; the lanes of a warp cover 512 contiguous bytes
          if (srow < tile_stride && q < p.Lq && p.tanh_ld) {   // window: the central samples only, straight to the caller
            for (int i = 0; i < p.tanh_cols; ++i) {
              const int n = q * p.tanh_cols + i;
              if (n >= p.tanh_s0 && n < p.tanh_s1) p.out_f32[(long long)b * p.tanh_ld + (n - p.tanh_s0)] = tanhf(v[i]);
            }
          } else if (srow < tile_stride && q < p.Lq) {
            float* dst = p.out_f32 + ((long long)b * p.Lq + q) * p.tanh_cols;
            if (p.tanh_cols == 4) {
              *reinterpret_cast<float4*>(dst) = make_float4(tanhf(v[0]), tanhf(v[1]), tanhf(v[2]), tanhf(v[3]));
            } else if (p.tanh_cols == 2) {
              *reinterpret_cast<float2*>(dst) = make_float2(tanhf(v[0]), tanhf(v[1]));
            } else {
              for (int i = 0; i < p.tanh_cols; ++i) dst[i] = tanhf(v[i]);
            }
          }
        }
        if (out_f32) {   // debug / parity hook only: plain per-thread stores
          const int n = q * p.out_stride + p.out_phase;
          const int oc_total = (MODE == EPI_TC_GATE) ? p.Cout / 2 : p.Cout;
          if (srow < tile_stride && q < p.Lq && n < p.Lout && och < oc_total) {
            float4* dst = reinterpret_cast<float4*>(out_f32 + ((long long)b * p.Lout + n) * oc_total + och);
#pragma unroll
            for (int i = 0; i < OW / 4; ++i) dst[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
          }
        }
        if (has_out) {
          const uint32_t row_off_out = (uint32_t)srow * (OW * 2);
          if (has_raw) stage_out<OW>(v, raw_b + ob, row_off_out, swz_out, n_parts, part_bytes);
          if (has_act) {
            if (n_parts == 1) {
              stage_out_act<OW>(v, act_b + ob, row_off_out, swz_out, slope);
            } else {
#pragma unroll
              for (int i = 0; i < OW; ++i) v[i] = fmaxf(v[i], v[i] * slope);   // leaky_relu, 0 < slope < 1
              stage_out<OW>(v, act_b + ob, row_off_out, swz_out, n_parts, part_bytes);
            }
          }
        }
      }
      if (has_out) {
        fence_async_smem();                // generic-proxy writes -> visible to the TMA (async proxy)
        // the previous unit's store (issued a whole unit ago) has finished reading its staging buffer: after this barrier
        // every warp may overwrite that buffer, which is the one the NEXT unit uses
        if (lead && elect_one()) bulk_wait_read<0>();
      }
      epi_bar_sync(2, epi_threads);        // barrier B: staging tile complete; add buffer fully consumed
      if (has_add) { if (++add_buf == n_add_bufs) add_buf = 0; }
      if (has_out) {
        if (lead && elect_one()) {     // elect.sync is deterministic: the same lane owns every bulk group
          for (int pt = 0; pt < n_parts; ++pt)
            for (int bx = 0; bx < e_n_boxes; ++bx) {
              const uint32_t off = ob + pt * part_bytes + bx * out_box_bytes;
              if (has_raw) tma_store_3d(&tmRaw, raw_b + off, och + pt * part_coff, tile_row0 + bx * e_box_rows, b);
              if (has_act) tma_store_3d(&tmAct, act_b + off, och + pt * part_coff, tile_row0 + bx * e_box_rows, b);
            }
          bulk_commit();
        }
        ++out_count;
      }
    }
    if (++as == 2) { as = 0; pacc ^= 1; }
  }
  if (lead && elect_one()) bulk_wait_all();
}

// The MMA issue loop is executed by a whole, converged warp: every operand is warp-uniform (kernel parameters, loop
// counters, the shuffled warp index / TMEM base), so the loop compiles to uniform-datapath code with back-to-back
// UTCHMMA instructions and the tensor pipe, not the issuing thread, sets the pace (tools/mma_bench2.cu: 40 / 48 / 64
// cycles per M=128 MMA at N <= 32 / 64 / 128).  Issued from a single-lane region the same loop cost ~80 cycles per MMA.
template <bool HALO, bool RESIDENT, int KK>
__device__ __forceinline__ void conv_tc_mma_loop(const ConvTC& p, uint32_t a_base, uint32_t w_base, uint32_t bar_base,
                                                 uint32_t tmem_base, int issuer, int n_issuers) {
  using namespace tc;
  const int total_tiles = p.total_tiles, n_achunks = p.n_achunks, ktaps = p.ktaps, stages_a = p.stages_a,
            stages_w = p.stages_w, n_tile = p.n_tile, mb = p.mb;
  int* const error_flag = p.error_flag;
  const uint32_t idesc = make_idesc_bf16(128, (uint32_t)n_tile);
  // descriptor words: hi = SBO | version | layout (constant), lo = LBO(1) << 16 | (address >> 4)
  const uint32_t desc_hi = ((p.sbo_bytes >> 4) & 0x3FFFu) | (1u << 14) | ((p.swizzle_code & 7u) << 29);
  const uint32_t lo_const = 1u << 16;
  const uint32_t a_lo0 = (a_base >> 4), w_lo0 = (w_base >> 4);
  const uint32_t a_stage16 = p.a_stage_bytes >> 4, w_stage16 = p.w_stage_bytes >> 4;
  const uint32_t tap_step16 = HALO ? (uint32_t)(p.dil * p.KC * 2) >> 4 : 0u;
  const uint32_t blk_step16 = (uint32_t)(128 * p.KC * 2) >> 4;     // one 128-row block further down the A tile
  bar_base += 8u * (uint32_t)p.bar_slot0;
  tmem_base += (uint32_t)p.tmem_col0;
  const uint32_t bar_a_full = bar_base + 8u * kBarAFull, bar_a_empty = bar_base + 8u * kBarAEmpty;
  const uint32_t bar_w_full = bar_base + 8u * kBarWFull, bar_w_empty = bar_base + 8u * kBarWEmpty;
  const uint32_t bar_acc_full = bar_base + 8u * kBarAccFull, bar_acc_empty = bar_base + 8u * kBarAccEmpty;
  auto mk = [&](uint32_t lo16) { return ((uint64_t)desc_hi << 32) | (uint64_t)(lo_const | (lo16 & 0x3FFFu)); };

  int sa = 0, sw = 0, as = 0;
  uint32_t pa = 0, pw = 0, pacc = 0;
  if (RESIDENT) mbar_wait(bar_w_full, 0, error_flag);
  for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
    mbar_wait(bar_acc_empty + 8u * as, pacc ^ 1, error_flag);
    fence_after_sync();
    const uint32_t d_tmem0 = tmem_base + (uint32_t)(as * mb * n_tile);
    uint32_t w_res16 = w_lo0;   // RESIDENT: walks the (chunk, pass, tap) tiles in order
    uint32_t first = 1;
    for (int c = 0; c < n_achunks; ++c) {
      if (HALO) { mbar_wait(bar_a_full + 8u * sa, pa, error_flag); fence_after_sync(); }
      const int n_wp = p.n_wpass[c];
      for (int wp = 0; wp < n_wp; ++wp) {
        uint32_t a16 = a_lo0 + (uint32_t)sa * a_stage16;
        for (int j = 0; j < ktaps; ++j) {
          if (!HALO) {
            mbar_wait(bar_a_full + 8u * sa, pa, error_flag);
            a16 = a_lo0 + (uint32_t)sa * a_stage16;
          }
          uint32_t w16;
          if (RESIDENT) { w16 = w_res16; w_res16 += w_stage16; }
          else { mbar_wait(bar_w_full + 8u * sw, pw, error_flag); w16 = w_lo0 + (uint32_t)sw * w_stage16; }
          if (!HALO || !RESIDENT) fence_after_sync();
          const uint32_t accumulate = first ? 0u : 1u;
          first = 0;
          uint32_t ab16 = a16 + (uint32_t)issuer * blk_step16, d_tmem = d_tmem0 + (uint32_t)(issuer * n_tile);
          for (int bi = issuer; bi < mb; bi += n_issuers) {   // every weight tile feeds mb MMAs, split over the issuers
#pragma unroll
            for (int kk = 0; kk < KK; ++kk) {
              // HALO: the row-shifted start address keeps base_offset = 0 -- the UMMA unit applies the swizzle
              // XOR to absolute shared-memory address bits (verified on B200, tools/tc_probe.py).
              if (elect_one()) umma_bf16(d_tmem, mk(ab16 + 2u * kk), mk(w16 + 2u * kk), idesc, (kk > 0) ? 1u : accumulate);
            }
            ab16 += blk_step16 * (uint32_t)n_issuers;
            d_tmem += (uint32_t)(n_tile * n_issuers);
          }
          if (HALO) a16 += tap_step16;
          if (!RESIDENT) {
            if (elect_one()) umma_commit(bar_w_empty + 8u * sw);
            if (++sw == stages_w) { sw = 0; pw ^= 1; }
          }
          if (!HALO) {
            if (elect_one()) umma_commit(bar_a_empty + 8u * sa);
            if (++sa == stages_a) { sa = 0; pa ^= 1; }
          }
        }
      }
      if (HALO) {
        if (elect_one()) umma_commit(bar_a_empty + 8u * sa);
        if (++sa == stages_a) { sa = 0; pa ^= 1; }
      }
    }
    if (elect_one()) umma_commit(bar_acc_full + 8u * as);
    if (++as == 2) { as = 0; pacc ^= 1; }
  }
}

// SMALL = true: the low-channel instantiation (epilogue chunks of <= 32 channels): register budget for TWO
// resident CTAs per SM, which doubles the single-thread MMA issue rate and the epilogue warps in flight.
template <bool SMALL, int SIG = EPI_SIG_GENERIC>
__global__ void __launch_bounds__(tc::kThreads, SMALL ? 2 : 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
               const __grid_constant__ CUtensorMap tmAdd0, const __grid_constant__ CUtensorMap tmAdd1,
               const __grid_constant__ CUtensorMap tmRaw, const __grid_constant__ CUtensorMap tmAct, const ConvTC p) {
  using namespace tc;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t a_base = smem_base + p.a_off;
  const uint32_t w_base = smem_base + p.w_off;
  const uint32_t bar_base = smem_base + p.bar_off;
  auto a_full = [&](int s) { return bar_base + 8u * (kBarAFull + s); };
  auto a_empty = [&](int s) { return bar_base + 8u * (kBarAEmpty + s); };
  auto w_full = [&](int s) { return bar_base + 8u * (kBarWFull + s); };
  auto w_empty = [&](int s) { return bar_base + 8u * (kBarWEmpty + s); };
  auto acc_full = [&](int s) { return bar_base + 8u * (kBarAccFull + s); };
  auto acc_empty = [&](int s) { return bar_base + 8u * (kBarAccEmpty + s); };
  const uint32_t tmem_slot = bar_base + 8u * kNumBars;
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // warp-uniform for the compiler

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmW);
    if (p.has_add0) prefetch_tmap(&tmAdd0);
    if (p.has_add1) prefetch_tmap(&tmAdd1);
    if (p.has_raw) prefetch_tmap(&tmRaw);
    if (p.has_act) prefetch_tmap(&tmAct);
    const uint32_t n_iss = p.mb >= 2 ? 2u : 1u;      // every issuer commits to the stage / accumulator barriers
    for (int s = 0; s < kMaxStages; ++s) {
      mbar_init(a_full(s), 1); mbar_init(a_empty(s), n_iss);
      mbar_init(w_full(s), 1); mbar_init(w_empty(s), n_iss);
    }
    for (int s = 0; s < 2; ++s) { mbar_init(acc_full(s), n_iss); mbar_init(acc_empty(s), p.epi_sets > 1 ? 8 : 4); }
    for (int s = 0; s < kMaxAddBufs; ++s) mbar_init(bar_base + 8u * (kBarAdd + s), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(tmem_slot, p.tmem_cols);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot_ptr, 0);
  // Programmatic dependent launch: let the next kernel of the stream start its prologue while this one runs, and do
  // not touch anything the previous kernel produced (activations, residuals, output buffers) before it has completed.
  // Only the resident-weight fetch below is independent of the previous kernel and is issued ahead of the wait.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (warp == 0 && lane == 0 && p.w_resident) {   // n_ntiles == 1: the weights do not depend on the tile
    mbar_expect_tx(w_full(0), (uint32_t)p.n_wtiles * p.w_box_bytes);
    int wt = 0;
    for (int c = 0; c < p.n_achunks; ++c)
      for (int wp = 0; wp < p.n_wpass[c]; ++wp)
        for (int j = 0; j < p.ktaps; ++j, ++wt)
          tma_load_2d(w_base + (uint32_t)wt * p.w_stage_bytes, &tmW, w_full(0), p.w_coff[c][wp], j * p.CoutT);
  }
  asm volatile("griddepcontrol.wait;" ::: "memory");

  if (warp == 0) {
    // ===================== TMA producer (converged warp, one elected lane per instruction) =====================
    {
      int sa = 0, sw = 0;
      uint32_t pa = 0, pw = 0;
      TileIter it;
      it.init((int)blockIdx.x, (int)gridDim.x, p.n_ntiles, p.m_tiles_per_b);
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, it.next()) {
        const int nt = it.nt, mt = it.mt, b = it.b;
        const int row0 = mt * p.tile_stride + p.in_off0;
        for (int c = 0; c < p.n_achunks; ++c) {
          if (p.halo_mode) {
            mbar_wait(a_empty(sa), pa ^ 1, p.error_flag);
            if (elect_one()) {
              mbar_expect_tx(a_full(sa), (uint32_t)p.a_n_boxes * p.a_box_bytes);
              for (int bx = 0; bx < p.a_n_boxes; ++bx)
                tma_load_3d(a_base + sa * p.a_stage_bytes + bx * p.a_box_bytes, &tmA, a_full(sa), p.a_coff[c],
                            row0 + bx * p.a_box_rows, b);
            }
            if (++sa == p.stages_a) { sa = 0; pa ^= 1; }
            if (p.w_resident) continue;
          }
          for (int wp = 0; wp < p.n_wpass[c]; ++wp) {
            for (int j = 0; j < p.ktaps; ++j) {
              if (!p.halo_mode) {   // RELOAD mode: mb == 1, one 128-row box per (chunk, pass, tap)
                mbar_wait(a_empty(sa), pa ^ 1, p.error_flag);
                if (elect_one()) {
                  mbar_expect_tx(a_full(sa), p.a_box_bytes);
                  tma_load_3d(a_base + sa * p.a_stage_bytes, &tmA, a_full(sa), p.a_coff[c], row0 + j * p.dil, b);
                }
                if (++sa == p.stages_a) { sa = 0; pa ^= 1; }
              }
              if (!p.w_resident) {
                mbar_wait(w_empty(sw), pw ^ 1, p.error_flag);
                if (elect_one()) {
                  mbar_expect_tx(w_full(sw), p.w_box_bytes);
                  tma_load_2d(w_base + sw * p.w_stage_bytes, &tmW, w_full(sw), p.w_coff[c][wp], j * p.CoutT + nt * p.n_tile);
                }
                if (++sw == p.stages_w) { sw = 0; pw ^= 1; }
              }
            }
          }
        }
      }
    }
  } else if (warp == 1 || warp == 6) {
    // ===================== MMA issuers =====================
    const int n_issuers = p.mb >= 2 ? 2 : 1;
    const int issuer = warp == 1 ? 0 : 1;
    if (issuer < n_issuers) {   // the whole warp runs the issue loop (see conv_tc_mma_loop)
      const int kk_n = p.KC / 16;
#define VSG_MMA(H, R)                                                                                        \
  do {                                                                                                       \
    if (kk_n == 4) conv_tc_mma_loop<H, R, 4>(p, a_base, w_base, bar_base, tmem_base, issuer, n_issuers);     \
    else if (kk_n == 2) conv_tc_mma_loop<H, R, 2>(p, a_base, w_base, bar_base, tmem_base, issuer, n_issuers); \
    else conv_tc_mma_loop<H, R, 1>(p, a_base, w_base, bar_base, tmem_base, issuer, n_issuers);               \
  } while (0)
      if (p.halo_mode && p.w_resident) VSG_MMA(true, true);
      else if (p.halo_mode) VSG_MMA(true, false);
      else if (p.w_resident) VSG_MMA(false, true);
      else VSG_MMA(false, false);
#undef VSG_MMA
    }
  } else {
    // ===================== epilogue (1 or 2 sets of 4 warps, one TMEM lane quarter per warp) =====================
    const int set = warp >= 7 ? 1 : 0, lead_warp = 2;
#define VSG_EPI(CWV)                                                                                              \
  do {                                                                                                            \
    if (p.mode == EPI_TC_LINEAR && p.n_parts == 2)                                                                \
      conv_tc_epilogue<CWV, EPI_TC_LINEAR, 2>(tmAdd0, tmAdd1, tmRaw, tmAct, p, smem_base, bar_base, tmem_base, warp, lane, set, lead_warp); \
    else if (p.mode == EPI_TC_LINEAR)                                                                             \
      conv_tc_epilogue<CWV, EPI_TC_LINEAR, 1>(tmAdd0, tmAdd1, tmRaw, tmAct, p, smem_base, bar_base, tmem_base, warp, lane, set, lead_warp); \
    else if (p.mode == EPI_TC_GATE)                                                                               \
      conv_tc_epilogue<CWV, EPI_TC_GATE, 1>(tmAdd0, tmAdd1, tmRaw, tmAct, p, smem_base, bar_base, tmem_base, warp, lane, set, lead_warp);   \
    else                                                                                                          \
      conv_tc_epilogue<CWV, EPI_TC_COUPLE, 1>(tmAdd0, tmAdd1, tmRaw, tmAct, p, smem_base, bar_base, tmem_base, warp, lane, set, lead_warp); \
  } while (0)
    if constexpr (SIG == EPI_SIG_GENERIC) {
      if (!SMALL && p.cw == 64) VSG_EPI(64);
      else if (p.cw == 32) VSG_EPI(32);
      else VSG_EPI(16);
    } else if constexpr (SIG == EPI_SIG_X6) {   // three planes per tensor: chunks of 32 / 16 channels (staging = 3 x the plain size)
#define VSG_EPI6(CWV)                                                                                             \
  do {                                                                                                            \
    if (p.mode == EPI_TC_LINEAR)                                                                                  \
      conv_tc_epilogue<CWV, EPI_TC_LINEAR, 3, SIG>(tmAdd0, tmAdd1, tmRaw, tmAct, p, smem_base, bar_base, tmem_base, warp, lane, set, lead_warp); \
    else if (p.mode == EPI_TC_GATE)                                                                               \
      conv_tc_epilogue<CWV, EPI_TC_GATE, 3, SIG>(tmAdd0, tmAdd1, tmRaw, tmAct, p, smem_base, bar_base, tmem_base, warp, lane, set, lead_warp);   \
    else                                                                                                          \
      conv_tc_epilogue<CWV, EPI_TC_COUPLE, 3, SIG>(tmAdd0, tmAdd1, tmRaw, tmAct, p, smem_base, bar_base, tmem_base, warp, lane, set, lead_warp); \
  } while (0)
      if (p.cw == 32) VSG_EPI6(32);
      else VSG_EPI6(16);
#undef VSG_EPI6
    } else if constexpr (SIG == EPI_SIG_ACT_X3 || SIG == EPI_SIG_RES_ACT_X3 || SIG == EPI_SIG_SUM0_X3 || SIG == EPI_SIG_SUM1_X3 ||
                         SIG == EPI_SIG_FINAL_X3) {
      if (!SMALL && p.cw == 64)
        conv_tc_epilogue<64, EPI_TC_LINEAR, 2, SIG>(tmAdd0, tmAdd1, tmRaw, tmAct, p, smem_base, bar_base, tmem_base, warp, lane, set, lead_warp);
      else if (p.cw == 32)
        conv_tc_epilogue<32, EPI_TC_LINEAR, 2, SIG>(tmAdd0, tmAdd1, tmRaw, tmAct, p, smem_base, bar_base, tmem_base, warp, lane, set, lead_warp);
      else
        conv_tc_epilogue<16, EPI_TC_LINEAR, 2, SIG>(tmAdd0, tmAdd1, tmRaw, tmAct, p, smem_base, bar_base, tmem_base, warp, lane, set, lead_warp);
    } else if constexpr (SIG == EPI_SIG_MAG) {
      if (!SMALL && p.cw == 64)
        conv_tc_epilogue<64, EPI_TC_MAG, 1, SIG>(tmAdd0, tmAdd1, tmRaw, tmAct, p, smem_base, bar_base, tmem_base, warp, lane, set, lead_warp);
      else if (p.cw == 32)
        conv_tc_epilogue<32, EPI_TC_MAG, 1, SIG>(tmAdd0, tmAdd1, tmRaw, tmAct, p, smem_base, bar_base, tmem_base, warp, lane, set, lead_warp);
      else
        conv_tc_epilogue<16, EPI_TC_MAG, 1, SIG>(tmAdd0, tmAdd1, tmRaw, tmAct, p, smem_base, bar_base, tmem_base, warp, lane, set, lead_warp);
    } else if constexpr (SIG == EPI_SIG_POST) {
      conv_tc_epilogue<16, EPI_TC_TANH, 1, SIG>(tmAdd0, tmAdd1, tmRaw, tmAct, p, smem_base, bar_base, tmem_base, warp, lane, set, lead_warp);
    } else {   // specialised signature: plain-bf16 linear epilogue with compile-time feature flags
      if (!SMALL && p.cw == 64)
        conv_tc_epilogue<64, EPI_TC_LINEAR, 1, SIG>(tmAdd0, tmAdd1, tmRaw, tmAct, p, smem_base, bar_base, tmem_base, warp, lane, set, lead_warp);
      else if (p.cw == 32)
        conv_tc_epilogue<32, EPI_TC_LINEAR, 1, SIG>(tmAdd0, tmAdd1, tmRaw, tmAct, p, smem_base, bar_base, tmem_base, warp, lane, set, lead_warp);
      else
        conv_tc_epilogue<16, EPI_TC_LINEAR, 1, SIG>(tmAdd0, tmAdd1, tmRaw, tmAct, p, smem_base, bar_base, tmem_base, warp, lane, set, lead_warp);
    }
#undef VSG_EPI
  }

  // ---- teardown: everyone done with TMEM before the allocating warp frees it ----
  fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    fence_after_sync();
    tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// ---- glue kernels of the bf16 path --------------------------------------------------------------

// [B, C, T] fp32 (reference layout) -> [B, T, planes * C] bf16 (channels-last).  32x32 smem tile.
// planes = 2: rows are [hi (C) | lo (C)] with hi = bf16(x), lo = bf16(x - hi)  (split-bf16 mode);
// planes = 3: [hi | mid | lo], the fp32 value exactly (the flow at the fp32 tolerance).
// ps_logs != null: x is mu_p and the value laid out is the prior sample z_p = (mu_p + noise * exp(logs_p)) * mask
// (models/visinger.py:107; the arithmetic of prior_sample_kernel), so the hot path needs no fp32 z_p tensor at all.
// x_ld > 0: x (and ps_*) are frames [0, T) of rows of x_ld frames -- a streaming window read in place from the whole batch.
__global__ void transpose_to_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, int C, int T,
                                         int planes, const float* __restrict__ ps_logs = nullptr,
                                         const float* __restrict__ ps_noise = nullptr, const float* __restrict__ ps_mask = nullptr,
                                         int x_ld = 0) {
  const int ld = x_ld > 0 ? x_ld : T;
  __shared__ float tile[32][33];
  const int b = blockIdx.z, c0 = blockIdx.y * 32, t0 = blockIdx.x * 32;
  const int tx = threadIdx.x, ty = threadIdx.y;   // 32 x 8
  for (int i = ty; i < 32; i += 8) {
    const int c = c0 + i, t = t0 + tx;
    float v = 0.f;
    if (c < C && t < T) {
      const long long idx = ((long long)b * C + c) * ld + t;
      v = x[idx];
      if (ps_logs) v = (v + ps_noise[idx] * expf(ps_logs[idx])) * ps_mask[(long long)b * ld + t];
    }
    tile[i][tx] = v;
  }
  __syncthreads();
  const int W = planes * C;
  for (int i = ty; i < 32; i += 8) {
    const int t = t0 + i, c = c0 + tx;
    if (t < T && c < C) {
      float v = tile[tx][i];
      for (int pl = 0; pl < planes; ++pl) {
        const __nv_bfloat16 h = __float2bfloat16(v);
        y[((long long)b * T + t) * W + pl * C + c] = h;
        v -= __bfloat162float(h);
      }
    }
  }
}

// [B, C, T] fp32 -> [B, T, Cp] bf16 with channels [C, Cp) written as zeros (rows padded to the kernels' channel chunks).
__global__ void transpose_pad_to_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, int C, int Cp, int T) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, c0 = blockIdx.y * 32, t0 = blockIdx.x * 32;
  const int tx = threadIdx.x, ty = threadIdx.y;   // 32 x 8
  for (int i = ty; i < 32; i += 8) {
    const int c = c0 + i, t = t0 + tx;
    tile[i][tx] = (c < C && t < T) ? x[((long long)b * C + c) * T + t] : 0.f;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int t = t0 + i, c = c0 + tx;
    if (t < T && c < Cp) y[((long long)b * T + t) * Cp + c] = __float2bfloat16(tile[tx][i]);
  }
}

// z = (mu + noise * exp(logs)) * mask with mu / logs the channel halves of stats [B, 2C, T]   (encoder.py:96-97)
__global__ void posterior_sample_from_stats_kernel(const float* __restrict__ stats, const float* __restrict__ noise,
                                                   const float* __restrict__ mask, float* __restrict__ z, int C, int T,
                                                   long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long CT = (long long)C * T;
  const long long b = i / CT, r = i - b * CT;
  const int t = (int)(r % T);
  z[i] = (stats[b * 2 * CT + r] + noise[i] * expf(stats[b * 2 * CT + CT + r])) * mask[b * T + t];
}

// [B, T, planes * C] bf16 -> [B, C, T] fp32 (the planes of a value are summed); flip != 0 reverses the channel order
// (an odd number of Flips); mask != null: the output is multiplied by mask[b][t] (`z * mask`, models/visinger.py:109-111),
// mask rows mask_ld apart (0: T).
__global__ void transpose_from_bf16_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ y, int C, int T,
                                           int flip, int planes, const float* __restrict__ mask = nullptr, int mask_ld = 0) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, c0 = blockIdx.y * 32, t0 = blockIdx.x * 32;
  const int tx = threadIdx.x, ty = threadIdx.y;   // 32 x 8
  for (int i = ty; i < 32; i += 8) {
    const int t = t0 + i, c = c0 + tx;
    float v = 0.f;
    if (c < C && t < T)
      for (int pl = 0; pl < planes; ++pl) v += __bfloat162float(x[((long long)b * T + t) * planes * C + pl * C + c]);
    tile[i][tx] = v;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int c = c0 + i, t = t0 + tx;
    if (c < C && t < T)
      y[((long long)b * C + (flip ? C - 1 - c : c)) * T + t] =
          mask ? tile[tx][i] * mask[(long long)b * (mask_ld > 0 ? mask_ld : T) + t] : tile[tx][i];
  }
}

// conv_post on the channels-last bf16 stream: input is already leaky_relu'd (out_act of the last stage).
// wav[b, n] = tanh(sum_{j, c} w[c][j] * x[b, n + j - pad, c]).  One thread per sample.
// split != 0: rows are [hi (C) | lo (C)] and x = hi + lo.  wav_ld > 0: only samples [n0, n1) are computed, into rows of
// wav wav_ld apart (a streaming window's central samples); else n0 = 0, n1 = L and the rows are L apart.
__global__ void conv_post_bf16_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ w /*[C][k]*/,
                                      float* __restrict__ wav, int C, int L, int k, int split, int n0 = 0, int n1 = 0,
                                      long long wav_ld = 0) {
  extern __shared__ float wsm[];   // [k][C]
  for (int i = threadIdx.x; i < C * k; i += blockDim.x) {
    const int c = i / k, j = i - c * k;
    wsm[j * C + c] = w[i];
  }
  __syncthreads();
  const int n = n0 + blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
  if (n >= (wav_ld ? n1 : L)) return;
  const int pad = (k - 1) / 2, W = split ? 2 * C : C;
  float s = 0.f;
  for (int j = 0; j < k; ++j) {
    const int pos = n + j - pad;
    if (pos < 0 || pos >= L) continue;
    const uint4* row = reinterpret_cast<const uint4*>(x + ((long long)b * L + pos) * W);
    for (int c8 = 0; c8 < C / 8; ++c8) {
      float f[8];
      tc::unpack_bf16x8(__ldg(row + c8), f);
      if (split) {
        float g2[8];
        tc::unpack_bf16x8(__ldg(row + C / 8 + c8), g2);
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] += g2[i];
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) s = fmaf(wsm[j * C + c8 * 8 + i], f[i], s);
    }
  }
  wav[wav_ld ? (long long)b * wav_ld + (n - n0) : (long long)b * L + n] = tanhf(s);
}

// conv_post for the shapes the model actually has (C = 16 channels, k = 7), plain bf16: every thread produces S
// consecutive samples from a sliding window of S + K - 1 input rows, so each row is fetched once per thread (two
// 16-byte loads at C = 16) and the inner loop is pure FFMA on weights the compiler keeps in registers / reloads from
// L1.  The one-thread-per-sample kernel above re-reads every row K times and spends one shared-memory load per FMA
// (165 us -> 94 us at B = 16, L = 300 000; HBM time is ~25 us).
template <int C, int K, int S>
__global__ void __launch_bounds__(128) conv_post_bf16_win_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ w /*[C][K]*/,
                                                                 float* __restrict__ wav, int L, int groups_per_b, int total_groups) {
  float wr[K][C];
#pragma unroll
  for (int c = 0; c < C; ++c)
#pragma unroll
    for (int j = 0; j < K; ++j) wr[j][c] = __ldg(w + c * K + j);
  constexpr int pad = (K - 1) / 2;
  for (int gidx = blockIdx.x * blockDim.x + threadIdx.x; gidx < total_groups; gidx += gridDim.x * blockDim.x) {
    const int b = gidx / groups_per_b, n0 = (gidx - b * groups_per_b) * S;
    const __nv_bfloat16* xb = x + (long long)b * L * C;
    float acc[S];
#pragma unroll
    for (int i = 0; i < S; ++i) acc[i] = 0.f;
#pragma unroll
    for (int r = 0; r < S + K - 1; ++r) {
      const int pos = n0 + r - pad;
      float f[C];
      if (pos >= 0 && pos < L) {
        const uint4* row = reinterpret_cast<const uint4*>(xb + (long long)pos * C);
#pragma unroll
        for (int c8 = 0; c8 < C / 8; ++c8) tc::unpack_bf16x8(__ldg(row + c8), f + 8 * c8);
      } else {
#pragma unroll
        for (int c = 0; c < C; ++c) f[c] = 0.f;
      }
#pragma unroll
      for (int i = 0; i < S; ++i) {
        const int j = r - i;                       // tap of sample i that reads this row
        if (j >= 0 && j < K) {
#pragma unroll
          for (int c = 0; c < C; ++c) acc[i] = fmaf(wr[j][c], f[c], acc[i]);
        }
      }
    }
    float* out = wav + (long long)b * L + n0;
#pragma unroll
    for (int i = 0; i < S; ++i)
      if (n0 + i < L) out[i] = tanhf(acc[i]);
  }
}

// The same computation with the input staged through shared memory: a CTA of 128 threads produces 128 * S consecutive
// samples of one utterance; the 128 * S + K - 1 input rows (C bf16 each) are fetched with fully coalesced 16-byte loads
// (the window kernel above has every lane 8 rows = 256 B apart: 32 sectors per load instruction, and the L1 pipe, not
// HBM, set its pace: 93 us for 173 MB) and every thread then slides its window over shared memory.  Rows are padded by
// 16 bytes per S rows so that the lanes' 16-byte reads fall into distinct banks.  wav_ld > 0: only samples [s0, s1) are
// stored, into rows of wav wav_ld apart (a streaming window's central samples).
template <int C, int K, int S>
__global__ void __launch_bounds__(128) conv_post_bf16_smem_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ w /*[C][K]*/,
                                                                  float* __restrict__ wav, int L, int tiles_per_b, int total_tiles,
                                                                  int s0 = 0, int s1 = 0, long long wav_ld = 0) {
  static_assert(C == 16 && S == 8, "layout below assumes 32-byte rows and 8 samples per thread");
  constexpr int TS = 128 * S;                    // samples per tile
  constexpr int ROWS = TS + K - 1;
  constexpr int pad = (K - 1) / 2;
  constexpr int V = C / 8;                       // 16-byte vectors per row
  __shared__ uint4 tile[ROWS * V + ROWS / S + 2];   // + one pad vector per S rows
  float wr[K][C];
#pragma unroll
  for (int c = 0; c < C; ++c)
#pragma unroll
    for (int j = 0; j < K; ++j) wr[j][c] = __ldg(w + c * K + j);
  for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
    const int b = t / tiles_per_b, n_tile0 = (t - b * tiles_per_b) * TS;
    const uint4* xb = reinterpret_cast<const uint4*>(x + (long long)b * L * C);
    __syncthreads();                             // the previous tile is fully consumed
    for (int i = threadIdx.x; i < ROWS * V; i += 128) {
      const int r = i / V, pos = n_tile0 - pad + r;
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (pos >= 0 && pos < L) v = __ldg(xb + (long long)pos * V + (i - r * V));
      tile[i + r / S] = v;
    }
    __syncthreads();
    const int r0 = threadIdx.x * S;              // my first row inside the tile
    float acc[S];
#pragma unroll
    for (int i = 0; i < S; ++i) acc[i] = 0.f;
#pragma unroll
    for (int r = 0; r < S + K - 1; ++r) {
      float f[C];
      const int rr = r0 + r;
      const uint4* row = tile + rr * V + rr / S;
#pragma unroll
      for (int c8 = 0; c8 < V; ++c8) tc::unpack_bf16x8(row[c8], f + 8 * c8);
#pragma unroll
      for (int i = 0; i < S; ++i) {
        const int j = r - i;
        if (j >= 0 && j < K) {
#pragma unroll
          for (int c = 0; c < C; ++c) acc[i] = fmaf(wr[j][c], f[c], acc[i]);
        }
      }
    }
    const int n0 = n_tile0 + r0;
    if (wav_ld) {
#pragma unroll
      for (int i = 0; i < S; ++i)
        if (n0 + i >= s0 && n0 + i < s1) wav[(long long)b * wav_ld + (n0 + i - s0)] = tanhf(acc[i]);
      continue;
    }
    float* out = wav + (long long)b * L + n0;
    if (n0 + S <= L && (((long long)b * L + n0) & 3) == 0) {
      reinterpret_cast<float4*>(out)[0] = make_float4(tanhf(acc[0]), tanhf(acc[1]), tanhf(acc[2]), tanhf(acc[3]));
      reinterpret_cast<float4*>(out)[1] = make_float4(tanhf(acc[4]), tanhf(acc[5]), tanhf(acc[6]), tanhf(acc[7]));
    } else {
#pragma unroll
      for (int i = 0; i < S; ++i)
        if (n0 + i < L) out[i] = tanhf(acc[i]);
    }
  }
}

}  // namespace vsg
