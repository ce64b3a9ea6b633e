// Self-attention of the relative-position transformer encoder on tcgen05 (bf16 mode; reference
// modules/rel_transformer.py:137-177, MultiHeadAttention.attention with window_size = 4, heads_share = True):
//   s_ij = (q_i . k_j + [|j-i| <= w] q_i . Ek[j-i+w]) / sqrt(dk);  s_ij = -1e4 where mask_i * mask_j == 0
//   p = softmax_j(s);  o_i = sum_j p_ij (v_j + [|j-i| <= w] Ev[j-i+w])
// One CTA = 128 queries of one (utterance, head); keys stream in tiles of 128.  Both GEMMs run on the 5th-gen tensor
// cores with TMEM accumulators, every operand arrives by TMA straight from the fused QKV projection's channels-last
// output [B, T, 3H]:
//   * S = Q K^T: A = Q tile, B = K tile, both K-major [128 rows x DK] as DK / CW swizzled chunks of CW channels
//     (CW = 32: SWIZZLE_64B; CW = 16: SWIZZLE_32B), accumulator 128 columns of TMEM, double-buffered;
//   * the relative-position key logits are one more small GEMM, Rq = Q Ek^T (N = 16), issued once per CTA;
//   * O += P V: A = P (bf16, written by the softmax warps into a swizzled K-major tile), B = the V tile EXACTLY as TMA
//     delivered it ([keys][d], i.e. MN-major for this product): the instruction descriptor's b_major bit and an MN-major
//     shared-memory descriptor (leading byte offset = chunk stride, stride byte offset = 8 key rows) make the tensor core
//     read it transposed -- no transposition pass anywhere.
// Softmax in two passes over the key tiles (pass 1: row maxima only; pass 2: p = exp2(s - m), row sums, P, O), so the
// O accumulator never has to be rescaled in tensor memory; the price is computing S twice, on a tensor pipe that is
// otherwise idle here.  Two sets of 4 softmax warps take alternate tile visits (each owns one S buffer and one P buffer);
// a thread owns one query row (its TMEM lane): row reductions need no shuffles.
// Warp roles (320 threads): 0 TMA producer, 1 TMEM allocator + MMA issuer, 2..9 softmax sets 0 / 1 (warp % 4 = TMEM lane
// quarter).  Every barrier wait is bounded (trap + error flag).
// Split-key mode (T > 2048, or any T through the debug hook): the keys are cut into chunks of chunk_tiles tiles at fixed
// multiples of the chunk size from key 0, and one CTA runs the two passes above over one (query tile, head, utterance,
// key chunk).  Key indices, the >= T test and the diagonal offset stay absolute, so a relative-position window that
// straddles a chunk border contributes to each chunk the weights of that chunk's keys.  Instead of normalising, set 0
// writes the chunk's unnormalised output (including the relative-value term), row maximum (exp2 domain) and row sum;
// attention_combine_kernel merges the chunks.
#pragma once
#include "conv_tc.cuh"
#include "rb_tc.cuh"

namespace vsg {

struct AttnTC {
  int B, T, n_heads, w;
  int n_tiles;                    // ceil(T / 128): key tiles (= query tiles)
  int chunk_tiles;                // key tiles per CTA (<= kAtMaxTiles); blockIdx.x = query tile + n_tiles * key chunk
  const float* mask;              // [B, T]
  const float* Ek;                // fp32 [2w+1][DK]
  const float* Ev;
  __nv_bfloat16* o;               // [B, T, n_heads * DK]
  float* o_part;                  // split-key mode (else null): fp32 [chunks][B][T][n_heads * DK] unnormalised output,
  float* m_part;                  //   [chunks][B][n_heads][T] row maxima (exp2 domain)
  float* l_part;                  //   [chunks][B][n_heads][T] row sums
  int* error_flag;
};

namespace tc {
constexpr int kAtQFull = 0, kAtKFull = 1, kAtKEmpty = 3, kAtVFull = 5, kAtVEmpty = 7, kAtSFull = 9, kAtSEmpty = 11,
              kAtPFull = 13, kAtPEmpty = 15, kAtOFull = 17, kAtNumBars = 18;
constexpr int kAtThreads = 320;
constexpr int kAtMaxTiles = 16;   // key tiles of one CTA: T <= 2048 in one launch, the key-chunk size of the split mode
}  // namespace tc

template <int DK>
struct AttnSmem {
  static constexpr int CW = DK % 32 == 0 ? 32 : 16;           // channels per swizzled chunk
  static constexpr int NCH = DK / CW;
  static constexpr uint32_t CHB = 128u * CW * 2u;             // one chunk of a 128-row tile
  static constexpr uint32_t TILEB = NCH * CHB;                // = 128 * DK * 2
  static constexpr uint32_t q_off = 0, k_off = TILEB, v_off = 3 * TILEB, p_off = 5 * TILEB;
  static constexpr uint32_t ek_off = p_off + 2 * 32768u;      // NCH chunks of [16 rows x CW] bf16
  static constexpr uint32_t EKB = NCH * 16u * CW * 2u;
  static constexpr uint32_t misc_off = (ek_off + EKB + 1023u) & ~1023u;
  // misc (floats): rel [128][16] | pw [2][128][16] | mx [2][128] | ls [2][128] | kmask u32 [kAtMaxTiles][4] | bars
  static constexpr uint32_t rel_off = misc_off, pw_off = rel_off + 128 * 16 * 4, mx_off = pw_off + 2 * 128 * 16 * 4,
                            ls_off = mx_off + 2 * 128 * 4, km_off = ls_off + 2 * 128 * 4,
                            bar_off = km_off + tc::kAtMaxTiles * 4 * 4, end = bar_off + 8 * tc::kAtNumBars + 16;
  static constexpr size_t bytes = end + 1024;                  // + alignment slack
};

template <int DK>
__global__ void __launch_bounds__(tc::kAtThreads, 1)
relenc_attention_tc_kernel(const __grid_constant__ CUtensorMap tmQKV, const AttnTC p) {
  using namespace tc;
  using SM = AttnSmem<DK>;
  constexpr int CW = SM::CW, NCH = SM::NCH, KS = CW / 16;
  constexpr uint32_t CHB = SM::CHB, TILEB = SM::TILEB;
  constexpr uint32_t kSwz = CW == 32 ? 4u : 6u;               // UMMA layout type: SWIZZLE_64B / SWIZZLE_32B
  constexpr uint32_t kSwzMask = CW == 32 ? 3u : 1u;
  constexpr uint32_t kSbo = 8u * CW * 2u;                     // 8 rows of a chunk
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* const sgen = smem_raw + (sbase - smem_u32(smem_raw));
  auto bar = [&](int slot) { return sbase + SM::bar_off + 8u * (uint32_t)slot; };
  const uint32_t tmem_slot = sbase + SM::bar_off + 8u * kAtNumBars;
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(sgen + SM::bar_off + 8u * kAtNumBars);
  float* const rel_s = reinterpret_cast<float*>(sgen + SM::rel_off);
  float* const pw_s = reinterpret_cast<float*>(sgen + SM::pw_off);
  float* const mx_s = reinterpret_cast<float*>(sgen + SM::mx_off);
  float* const ls_s = reinterpret_cast<float*>(sgen + SM::ls_off);
  uint32_t* const km_s = reinterpret_cast<uint32_t*>(sgen + SM::km_off);
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int b = blockIdx.z, h = blockIdx.y, kc = blockIdx.x / p.n_tiles, q0 = (blockIdx.x - kc * p.n_tiles) * 128;
  const int kt0 = kc * p.chunk_tiles;                           // first key tile of this CTA's chunk
  const int T = p.T, H = p.n_heads * DK, nt = min(p.chunk_tiles, p.n_tiles - kt0), w = p.w, nrel = 2 * w + 1;
  int* const error_flag = p.error_flag;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmQKV);
    mbar_init(bar(kAtQFull), 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(bar(kAtKFull + s), 1); mbar_init(bar(kAtKEmpty + s), 1);
      mbar_init(bar(kAtVFull + s), 1); mbar_init(bar(kAtVEmpty + s), 1);
      mbar_init(bar(kAtSFull + s), 1); mbar_init(bar(kAtSEmpty + s), 4);
      mbar_init(bar(kAtPFull + s), 4); mbar_init(bar(kAtPEmpty + s), 1);
    }
    mbar_init(bar(kAtOFull), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  // Ek -> bf16 K-major chunks [16 rows x CW] (rows >= 2w+1 zero), swizzled like a TMA box; pw / key-mask words
  for (int i = threadIdx.x; i < 16 * DK; i += blockDim.x) {
    const int r = i / DK, d = i % DK, c = d / CW, dc = d % CW;
    const float v = r < nrel ? p.Ek[r * DK + d] : 0.f;
    const uint32_t off = (uint32_t)c * (16u * CW * 2u) + (uint32_t)r * (CW * 2u) + (uint32_t)dc * 2u;
    *reinterpret_cast<__nv_bfloat16*>(sgen + SM::ek_off + swz(off, kSwzMask)) = __float2bfloat16(v);
  }
  for (int i = threadIdx.x; i < 2 * 128 * 16; i += blockDim.x) pw_s[i] = 0.f;
  for (int i = warp; i < nt * 4; i += (int)(blockDim.x >> 5)) {
    const int t = (kt0 * 4 + i) * 32 + lane;
    const uint32_t bits = __ballot_sync(0xffffffffu, t < T && p.mask[(long long)b * T + t] != 0.f);
    if (lane == 0) km_s[i] = bits;
  }
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot_ptr, 0);
  const uint32_t tm_s = tmem_base, tm_o = tmem_base + 256u, tm_rq = tmem_base + 384u;
  const int n_visits = 2 * nt;                                  // pass 1 (maxima), then pass 2 (P, O)

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      mbar_expect_tx(bar(kAtQFull), TILEB);
      for (int c = 0; c < NCH; ++c) tma_load_3d(sbase + SM::q_off + c * CHB, &tmQKV, bar(kAtQFull), h * DK + c * CW, q0, b);
    }
    for (int v = 0; v < n_visits; ++v) {
      const int s = v & 1, k0 = (kt0 + v % nt) * 128;
      mbar_wait(bar(kAtKEmpty + s), (((uint32_t)v >> 1) & 1u) ^ 1u, error_flag);
      if (elect_one()) {
        mbar_expect_tx(bar(kAtKFull + s), TILEB);
        for (int c = 0; c < NCH; ++c)
          tma_load_3d(sbase + SM::k_off + s * TILEB + c * CHB, &tmQKV, bar(kAtKFull + s), H + h * DK + c * CW, k0, b);
      }
      if (v >= nt) {
        const int u = v - nt, sv = u & 1;
        mbar_wait(bar(kAtVEmpty + sv), (((uint32_t)u >> 1) & 1u) ^ 1u, error_flag);
        if (elect_one()) {
          mbar_expect_tx(bar(kAtVFull + sv), TILEB);
          for (int c = 0; c < NCH; ++c)
            tma_load_3d(sbase + SM::v_off + sv * TILEB + c * CHB, &tmQKV, bar(kAtVFull + sv), 2 * H + h * DK + c * CW, k0, b);
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (converged warp) =====================
    constexpr uint32_t lo_flag = 1u << 16;                       // K-major descriptors: LBO field = 1 (unused)
    constexpr uint32_t hi_km = ((kSbo >> 4) & 0x3FFFu) | (1u << 14) | (kSwz << 29);          // Q / K / Ek chunks
    constexpr uint32_t hi_p = ((1024u >> 4) & 0x3FFFu) | (1u << 14) | (2u << 29);             // P: SWIZZLE_128B chunks of 64 keys
    // V as the MN-major B operand: LBO = stride between the CW-wide channel chunks, SBO = stride between groups of 8 keys
    constexpr uint32_t lbo_v = ((CHB >> 4) & 0x3FFFu) << 16;
    constexpr uint32_t hi_v = ((kSbo >> 4) & 0x3FFFu) | (1u << 14) | (kSwz << 29);
    auto mk = [&](uint32_t hi, uint32_t lo) { return ((uint64_t)hi << 32) | (uint64_t)lo; };
    const uint32_t idesc_s = make_idesc_bf16(128, 128), idesc_rq = make_idesc_bf16(128, 16);
    const uint32_t idesc_pv = make_idesc_bf16(128, (uint32_t)DK) | (1u << 16);               // b_major = MN
    const uint32_t q16 = (sbase + SM::q_off) >> 4, k16 = (sbase + SM::k_off) >> 4, v16 = (sbase + SM::v_off) >> 4,
                   p16 = (sbase + SM::p_off) >> 4, ek16 = (sbase + SM::ek_off) >> 4;
    constexpr uint32_t ch16 = CHB >> 4, tile16 = TILEB >> 4, ekch16 = (16u * CW * 2u) >> 4;
    uint32_t n_pv[2] = {0u, 0u};                                 // PV products issued per P buffer
    auto issue_pv = [&](int pv) {
      const int g = pv & 1, u = pv - nt, sv = u & 1;
      mbar_wait(bar(kAtPFull + g), n_pv[g] & 1u, error_flag);
      mbar_wait(bar(kAtVFull + sv), ((uint32_t)u >> 1) & 1u, error_flag);
      fence_after_sync();
      ++n_pv[g];
#pragma unroll
      for (int ks = 0; ks < 8; ++ks) {                           // 16 keys per step
        const uint32_t a_lo = lo_flag | (p16 + (uint32_t)g * 2048u + (uint32_t)(ks >> 2) * 1024u + (uint32_t)(ks & 3) * 2u);
        const uint32_t b_lo = lbo_v | (v16 + (uint32_t)sv * tile16 + (uint32_t)ks * (uint32_t)((16 * CW * 2) >> 4));
        if (elect_one()) umma_bf16(tm_o, mk(hi_p, a_lo), mk(hi_v, b_lo), idesc_pv, (u > 0 || ks > 0) ? 1u : 0u);
      }
      if (elect_one()) umma_commit(bar(kAtPEmpty + g));
      if (elect_one()) umma_commit(bar(kAtVEmpty + sv));
    };
    mbar_wait(bar(kAtQFull), 0u, error_flag);
    fence_after_sync();
#pragma unroll
    for (int c = 0; c < NCH; ++c)
#pragma unroll
      for (int kk = 0; kk < KS; ++kk)
        if (elect_one())
          umma_bf16(tm_rq, mk(hi_km, lo_flag | (q16 + c * ch16 + 2u * kk)), mk(hi_km, lo_flag | (ek16 + c * ekch16 + 2u * kk)),
                    idesc_rq, (c > 0 || kk > 0) ? 1u : 0u);
    for (int v = 0; v < n_visits; ++v) {
      const int s = v & 1;
      mbar_wait(bar(kAtKFull + s), ((uint32_t)v >> 1) & 1u, error_flag);
      mbar_wait(bar(kAtSEmpty + s), (((uint32_t)v >> 1) & 1u) ^ 1u, error_flag);
      fence_after_sync();
#pragma unroll
      for (int c = 0; c < NCH; ++c)
#pragma unroll
        for (int kk = 0; kk < KS; ++kk)
          if (elect_one())
            umma_bf16(tm_s + (uint32_t)s * 128u, mk(hi_km, lo_flag | (q16 + c * ch16 + 2u * kk)),
                      mk(hi_km, lo_flag | (k16 + (uint32_t)s * tile16 + c * ch16 + 2u * kk)), idesc_s, (c > 0 || kk > 0) ? 1u : 0u);
      if (elect_one()) umma_commit(bar(kAtSFull + s));
      if (elect_one()) umma_commit(bar(kAtKEmpty + s));
      if (v - 1 >= nt) issue_pv(v - 1);                          // the previous visit's P is ready by now (or soon)
    }
    issue_pv(n_visits - 1);
    if (elect_one()) umma_commit(bar(kAtOFull));
  } else {
    // ===================== softmax sets =====================
    const int g = (warp - 2) >> 2, quarter = warp & 3;
    const int row = quarter * 32 + lane, qi = q0 + row;
    const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
    const float sc2 = rsqrtf((float)DK) * 1.4426950408889634f;  // 1/sqrt(dk) * log2(e): scores live in the exp2 domain
    const float neg_fill = -1e4f * 1.4426950408889634f;
    const bool mq = qi < T && p.mask[(long long)b * T + qi] != 0.f;
    float* const my_rel = rel_s + row * 16;
    float* const my_pw = pw_s + (g * 128 + row) * 16;
    const uint32_t p_row = sbase + SM::p_off + (uint32_t)g * 32768u + (uint32_t)row * 128u;
    const uint32_t p_x = (uint32_t)(row & 7);
    float m_run = -INFINITY, l_run = 0.f;
    uint32_t n_s = 0, n_pw = 0;
    bool have_rel = false;
    // One visit = one key tile in one pass.  PASS2 = false: row maximum only; true: P, row sum, diagonal weights.
    auto visit = [&](int v, bool pass2) {
      const int k0 = (kt0 + v % nt) * 128;
      mbar_wait(bar(kAtSFull + g), n_s & 1u, error_flag);
      ++n_s;
      fence_after_sync();
      if (!have_rel) {                                           // Rq = Q Ek^T was issued ahead of the first S tile
        uint32_t r[16];
        tmem_ld16_nowait(tm_rq + lane_addr, r);
        tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < 16; ++i) my_rel[i] = __uint_as_float(r[i]) * sc2;   // (both sets write the same values)
        have_rel = true;
      }
      if (pass2 && n_pw > 0) mbar_wait(bar(kAtPEmpty + g), (n_pw - 1) & 1u, error_flag);   // my P buffer is free again
      const int d0 = qi - w - k0;                                // tile column of relative position -w
      float lsum = 0.f;
#pragma unroll 1
      for (int cc = 0; cc < 4; ++cc) {                           // 32 score columns at a time
        uint32_t r[32];
        tmem_ld16_nowait(tm_s + lane_addr + (uint32_t)(g * 128 + cc * 32), r);
        tmem_ld16_nowait(tm_s + lane_addr + (uint32_t)(g * 128 + cc * 32 + 16), r + 16);
        tmem_wait_ld();
        const uint32_t kw = km_s[(v % nt) * 4 + cc];
        const int c0 = cc * 32;
        const bool diag = d0 < c0 + 32 && d0 + nrel > c0;         // this chunk holds relative positions of my row
        float x[32];
#pragma unroll
        for (int e = 0; e < 32; ++e) x[e] = __uint_as_float(r[e]) * sc2;
        if (diag) {
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            const int d = c0 + e - d0;
            if ((unsigned)d < (unsigned)nrel) x[e] += my_rel[d];
          }
        }
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          if (!(mq && ((kw >> e) & 1u))) x[e] = neg_fill;        // masked_fill(mask == 0, -1e4)   (:167)
          if (k0 + c0 + e >= T) x[e] = -INFINITY;               // beyond the sequence: not a key at all
        }
        if (!pass2) {
#pragma unroll
          for (int e = 0; e < 32; ++e) m_run = fmaxf(m_run, x[e]);
        } else {
          uint32_t pk[16];
#pragma unroll
          for (int e = 0; e < 32; e += 2) {
            const float p0 = exp2f(x[e] - m_run), p1 = exp2f(x[e + 1] - m_run);
            lsum += p0 + p1;
            pk[e >> 1] = pack_bf16x2(p0, p1);
            x[e] = p0; x[e + 1] = p1;
          }
          if (diag) {
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              const int d = c0 + e - d0;
              if ((unsigned)d < (unsigned)nrel && k0 + c0 + e < T) my_pw[d] = x[e];
            }
          }
          const uint32_t chunk = p_row + (uint32_t)(cc >> 1) * 16384u;
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4)
            sts128(chunk + ((((uint32_t)(cc & 1) * 4u + (uint32_t)q4) ^ p_x) << 4),
                   make_uint4(pk[4 * q4], pk[4 * q4 + 1], pk[4 * q4 + 2], pk[4 * q4 + 3]));
        }
      }
      l_run += lsum;
      fence_before_sync();                                       // S buffer drained
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(kAtSEmpty + g));
      if (pass2) {
        fence_async_smem();                                      // P (generic writes) -> tensor core (async proxy)
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(kAtPFull + g));
        ++n_pw;
      }
    };
    for (int v = g; v < nt; v += 2) visit(v, false);
    // between the passes: the row maximum over ALL tiles (both sets)
    mx_s[g * 128 + row] = m_run;
    epi_bar_sync(1, 256);
    m_run = fmaxf(mx_s[row], mx_s[128 + row]);
    for (int v = nt + ((nt & 1) ^ g); v < n_visits; v += 2) visit(v, true);
    // ---- combine the two sets' row sums and diagonal weights; set 0 writes the output
    ls_s[g * 128 + row] = l_run;
    epi_bar_sync(2, 256);
    if (g == 0) {
      const float lsum = ls_s[row] + ls_s[128 + row];
      const float inv = 1.0f / lsum;
      if (p.o_part && qi < T) {
        const long long r = (((long long)kc * p.B + b) * p.n_heads + h) * T + qi;
        p.m_part[r] = m_run;
        p.l_part[r] = lsum;
      }
      mbar_wait(bar(kAtOFull), 0u, error_flag);
      fence_after_sync();
      __nv_bfloat16* orow = p.o + ((long long)b * T + qi) * H + h * DK;
#pragma unroll 1
      for (int c0 = 0; c0 < DK; c0 += 16) {
        uint32_t r[16];
        tmem_ld16_nowait(tm_o + lane_addr + (uint32_t)c0, r);
        tmem_wait_ld();
        float v[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
        for (int m = 0; m < nrel; ++m) {
          const float pm = pw_s[row * 16 + m] + pw_s[(128 + row) * 16 + m];
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = fmaf(pm, __ldg(p.Ev + m * DK + c0 + i), v[i]);
        }
        if (p.o_part) {
          float* orow32 = p.o_part + (((long long)kc * p.B + b) * T + qi) * H + h * DK + c0;
          if (qi < T)
#pragma unroll
            for (int i = 0; i < 16; i += 4) *reinterpret_cast<float4*>(orow32 + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
        } else if (qi < T) {
          uint32_t hh[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) hh[i] = pack_bf16x2(v[2 * i] * inv, v[2 * i + 1] * inv);
          stg128(orow + c0, make_uint4(hh[0], hh[1], hh[2], hh[3]));
          stg128(orow + c0 + 8, make_uint4(hh[4], hh[5], hh[6], hh[7]));
        }
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    fence_after_sync();
    tmem_dealloc(tmem_base, 512);
  }
}

// Merge of the split-key mode's chunks, one thread per 8 channels of one (utterance, frame):
//   M = max_c m_c;  w_c = exp2(m_c - M);  o = sum_c w_c o_c;  l = sum_c w_c l_c  (fmaf in chunk order from 0);  bf16(o / l)
// The chunk holding the maximum gets weight exactly 1 (one chunk reproduces the single-launch epilogue bit for bit); a
// chunk whose keys are all masked for a valid row has m_c = -1e4 log2(e) and weight exactly 0, and its finite o_c adds
// exactly 0, so masked padding leaves the result unchanged bit for bit.  A masked query row has m_c = -1e4 log2(e) in
// every chunk: weights 1, a uniform softmax over all T keys as in the reference.
__global__ void attention_combine_kernel(const float* __restrict__ o_part, const float* __restrict__ m_part,
                                         const float* __restrict__ l_part, __nv_bfloat16* __restrict__ o, int B, int T,
                                         int n_heads, int dk, int n_chunks) {
  using namespace tc;
  const int H = n_heads * dk, H8 = H / 8;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)B * T * H8) return;
  const long long bt = i / H8;                                  // b * T + t
  const int c = (int)(i - bt * H8) * 8, b = (int)(bt / T), t = (int)(bt - (long long)b * T), h = c / dk;
  const long long mrow = ((long long)b * n_heads + h) * T + t, mstride = (long long)B * n_heads * T;
  const long long orow = bt * H + c, ostride = (long long)B * T * H;
  float M = -INFINITY;
  for (int k = 0; k < n_chunks; ++k) M = fmaxf(M, m_part[k * mstride + mrow]);
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, l = 0.f;
  for (int k = 0; k < n_chunks; ++k) {
    const float wk = exp2f(m_part[k * mstride + mrow] - M);
    l = fmaf(wk, l_part[k * mstride + mrow], l);
    const float4 a = *reinterpret_cast<const float4*>(o_part + k * ostride + orow);
    const float4 d = *reinterpret_cast<const float4*>(o_part + k * ostride + orow + 4);
    const float x[8] = {a.x, a.y, a.z, a.w, d.x, d.y, d.z, d.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = fmaf(wk, x[j], acc[j]);
  }
  const float inv = 1.0f / l;
  uint32_t hh[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) hh[j] = pack_bf16x2(acc[2 * j] * inv, acc[2 * j + 1] * inv);
  stg128(o + orow, make_uint4(hh[0], hh[1], hh[2], hh[3]));
}

// fp32 workspace of the split-key mode: o_part, then m_part, then l_part (see AttnTC)
inline size_t attention_split_floats(int B, int T, int n_heads, int dk, int chunk_tiles) {
  const size_t n_chunks = (size_t)((T + 127) / 128 + chunk_tiles - 1) / chunk_tiles;
  return n_chunks * B * T * ((size_t)n_heads * dk + 2 * n_heads);
}

}  // namespace vsg
