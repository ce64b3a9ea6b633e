// bf16 tensor-core mode: weight pre-pack, TMA tensor maps, launch logic and the Generator driver.
#include <numeric>

#include "vsg_common.cuh"
#include "run.cuh"
#include "pack_tc.cuh"
#include "conv_tc.cuh"
#include "pair_tc.cuh"
#include "rb_tc.cuh"
#include "rp_tc.cuh"
#include "relenc_tc.cuh"
#include "attn_tc.cuh"
#include "spec.cuh"

#include <algorithm>
#include <map>
#include <mutex>
#include <utility>
#include <stdlib.h>

namespace vsg {

namespace {

// ---- cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time libcuda dependency) ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  });
  return fn;
}

CUtensorMapSwizzle swizzle_for(int kc) {
  return kc >= 64 ? CU_TENSOR_MAP_SWIZZLE_128B : kc >= 32 ? CU_TENSOR_MAP_SWIZZLE_64B
         : kc >= 16 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
}

int pick_kc(int cin) { return cin % 64 == 0 ? 64 : cin % 32 == 0 ? 32 : cin % 16 == 0 ? 16 : 0; }
// Largest UMMA N (multiple of 16, <= 256) that divides Cout and is itself a multiple of its epilogue chunk.
int pick_ntile(int cout) {
  if (cout % 16) return 0;
  for (int n = 256; n >= 16; n -= 16)
    if (cout % n == 0) return n;
  return 0;
}
int pick_cw(int nt) {
  if (nt >= 256) return 32;
  for (int c : {64, 32, 16})
    if (nt % c == 0) return c;
  return 16;
}

int encode_2d(CUtensorMap* m, const void* base, uint64_t inner, uint64_t rows, uint32_t box_inner, uint32_t box_rows,
              int kc) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(VSG_ECUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {inner, rows};
  cuuint64_t strides[1] = {inner * 2};
  cuuint32_t box[2] = {box_inner, box_rows};
  cuuint32_t es[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(kc), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(VSG_ECUDA, "cuTensorMapEncodeTiled(2d) failed with %d", (int)r);
  return VSG_OK;
}

// 3-D map over a channels-last bf16 tensor viewed as (C, rows, B) with explicit row / batch strides (elements).
int encode_3d(CUtensorMap* m, const void* base, uint64_t C, uint64_t rows, uint64_t B, uint64_t row_stride,
              uint64_t batch_stride, uint32_t box_c, uint32_t box_rows, int swz_elems) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(VSG_ECUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[3] = {C, rows, B};
  cuuint64_t strides[2] = {row_stride * 2, batch_stride * 2};
  cuuint32_t box[3] = {box_c, box_rows, 1};
  cuuint32_t es[3] = {1, 1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(swz_elems), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(VSG_ECUDA, "cuTensorMapEncodeTiled(3d) failed with %d", (int)r);
  return VSG_OK;
}

constexpr size_t kSmemMax = 227 * 1024;

struct EpiTC {
  int mode = EPI_TC_LINEAR;
  const float* mask = nullptr;      // [B][mask_ld]
  int mask_ld = 0;                  // 0: Lout
  int couple_sign = -1;
  int ld = 0;                       // leading dimension (channels per row) of the add / out tensors; 0 = their own width
  int part_stride = 0;              // channels between the bf16 planes of the add / out tensors; 0 = their own width
  int add0_is_act = 0;              // add0 holds leaky_relu(residual): invert it in the epilogue
  const float* bias = nullptr;
  const float* bcond = nullptr; int bcond_bs = 0;
  const __nv_bfloat16* add0 = nullptr;
  const __nv_bfloat16* add1 = nullptr;
  float scale = 1.f;
  float slope = 0.1f;               // leaky_relu slope of out_act (0 = ReLU)
  __nv_bfloat16* out_raw = nullptr;
  __nv_bfloat16* out_act = nullptr;
  float* out_f32 = nullptr;
  int tanh_cols = 0;                // EPI_TC_TANH: samples per row written to out_f32
  long long tanh_ld = 0;            // EPI_TC_TANH, > 0: only samples [tanh_s0, tanh_s1), at out_f32 + b * tanh_ld (conv_tc.cuh)
  int tanh_s0 = 0, tanh_s1 = 0;
  int mag_ch = 0;                   // EPI_TC_MAG: output channels below this are magnitudes, the rest are written as 0
};

// HALO mode verified on B200 (tools/tc_probe.py): the UMMA unit applies the swizzle XOR to absolute
// shared-memory address bits, so a row-shifted start address needs base_offset = 0.
struct TCOptions {
  int halo_mode = 1; int w_resident = 1; int max_mb = 4; int plan_only = 0;
  int force_mb = 0, force_cw = 0, force_two = -1, force_resident = -1;   // tuning overrides (0 / -1 = automatic)
  int use_pdl = 1;
  int fuse_pairs = 1;
  int merge_ups = 1;
  int split_n = 1;
  int single_stream = 1;
  int chain_streams = 1;
  int epi_sigs = 2;         // 0: one generic image; 1: ACT / RES_ACT / LINEAR images; 2: + SUM0 / SUM1 / FINAL
  int epi_sets = 2;
  int fuse_rb = 0;          // whole-ResBlock1 kernel (rb_tc.cuh) for the C <= 64 stages (opt-in: bit 15)
  int rb_max_mb = 0;        // cap on 128-row blocks per resblock tile (0 = as many as fit)
  int rb_sets = 4;          // epilogue warp sets of the resblock kernel
  int rb_issuers = 0;       // MMA issuer warps of the resblock kernel (0 = by channel count)
  int fuse_rp = 1;          // row-packed whole-ResBlock1 kernel (rp_tc.cuh) for the C <= 32 stages
  int rp_max_c = 32;        // widest stage the row-packed kernel takes
  int rp_packed = 1;        // dilation-1 convolutions in the block-Toeplitz form (0: every conv tap by tap)
  int rp_max_mb = 0;        // cap on 128-row blocks per row-packed tile (0 = as many as fit)
  int rp_two_cta = 0;       // row-packed kernel, plain bf16: two CTAs per SM (8 epilogue warps, 2-block tiles, streamed ring); bit 2
  int rp_x3 = 1;            // bf16x3 mode: the row-packed kernel's split-bf16 instantiation for the C <= 32 stages (bit 1: off)
  int rp_spb2 = 0;          // row-packed kernel, 3- / 4-block tiles: two epilogue warp sets per block, two blocks per set
                            // (measured slower: 314 / 415 / 513 us vs 289 / 386 / 491 at C = 32 -- the per-block hand-over, not the
                            // drain itself, is what a set spends its time on)
  int flow_merge = 1;       // flow: res_skip as one launch on the [h | out] tensor, every flow's cond_layer in one GEMV
  int conv_post = 0;        // conv_post kernel: 0 tcgen05 (row-packed, tanh epilogue), 1 register window, 2 shared-memory window
  uint32_t* rp_trace = nullptr;   // tuning aid (vsg_debug_resblock_bf16 with VSG_RP_TRACE set): pipeline event clocks of CTA 0
};

TCOptions g_default_opts;

constexpr size_t kSmemBudget = 227 * 1024 - 2048;   // dynamic smem we plan within (1 KB alignment slack + barriers)

struct TunedPlan { int cin, cout, k, n_adds, n_outs, x3, mb, cw, two, resident; };
static const TunedPlan kTunedPlans[] = {
#include "tc_plan_table.inc"
    {0, 0, 0, 0, 0, 0, 0, 0, 0, 0}};

// One convolution launch.  x: [B, Lin, Cin] bf16 channels-last; add/out tensors: [B, Lout, Cout].
int launch_conv_tc(const VsgPack* P, const ConvWTC& w, const __nv_bfloat16* x, int B, int Lin, int in_off0, int dil,
                   int Lq, int out_stride, int out_phase, int Lout, const EpiTC& e, const TCOptions& opt, int* error_flag,
                   cudaStream_t st, int x_ld = 0, int x_part_stride = 0, int* image_out = nullptr) {
  const int a_planes = w.wsplit ? 1 : w.planes;           // bf16 planes of the activations and of every epilogue tensor
  if (x_ld == 0) x_ld = a_planes * w.Cin;
  if (x_part_stride == 0) x_part_stride = w.Cin;          // channels between the bf16 planes of an input row
  if (w.planes == 2 && !w.wsplit && e.mode != EPI_TC_LINEAR) return fail(VSG_EUNSUPPORTED, "split-bf16 supports the linear epilogue only");
  if (!w.has_tmap) return fail(VSG_EUNSUPPORTED, "bf16 tensor-core path needs channel counts that are multiples of 16 "
                                                 "(conv %d -> %d)", w.Cin, w.Cout);
  if (Lq <= 0 || B <= 0) return VSG_OK;
  // a convolution with taps reads rows that other CTAs' output tiles cover: it must not write over its own input
  if (w.ktaps > 1 && ((const void*)x == (const void*)e.out_act || (const void*)x == (const void*)e.out_raw))
    return fail(VSG_EINVAL, "a k > 1 convolution must not run in place (output aliases the input)");
  const int KC = pick_kc(w.Cin);
  int NT = pick_ntile(w.Cout);                 // output-channel tile; N = 256 convs may also run as 2 x 128 (see below)
  const int halo = (w.ktaps - 1) * dil;
  const bool halo_ok = opt.halo_mode && 128 + halo <= 256;
  // low-channel convolutions run the SMALL kernel instantiation (<= 32-channel epilogue chunks, 2 CTAs / SM)
  bool small = NT <= 64 && (NT <= 32 || NT % 32 == 0);
  int cw_max = small ? std::min(NT, 32) : pick_cw(NT);
  if (w.planes == 3) cw_max = std::min(cw_max, 32);       // the three-plane epilogue is instantiated for 32 / 16 channels
  const bool pairs = e.mode == EPI_TC_GATE || e.mode == EPI_TC_MAG;   // two accumulator columns per output channel
  const int cout_eff = pairs ? w.Cout / 2 : w.Cout;  // channels of the add / out tensors
  const int n_parts = a_planes;
  const int part_stride = e.part_stride ? e.part_stride : cout_eff;
  const int ld = e.ld ? e.ld : n_parts * cout_eff;
  const int n_adds = (e.add0 ? 1 : 0) + (e.add1 ? 1 : 0), n_outs = (e.out_raw ? 1 : 0) + (e.out_act ? 1 : 0);
  const size_t half_budget = 110 * 1024;

  // Plan the tile: try mb = 4, 2, 1 blocks of 128 rows; prefer the largest that lets two CTAs share an SM (small
  // kernels), else the largest that fits at all.
  ConvTC p;
  auto plan = [&](int mb, int cw, size_t budget, int force_resident, ConvTC* out) -> bool {
    ConvTC q;
    memset(&q, 0, sizeof(q));
    if (NT % cw) return false;
    if (mb > 1 && !halo_ok) return false;
    if (2 * mb * NT > 512) return false;
    if (mb > 1 && Lq < 128 * mb) return false;
    q.mb = mb;
    q.KC = KC; q.ktaps = w.ktaps; q.dil = dil; q.in_off0 = in_off0;
    const int nc = w.Cin / KC;
    q.n_achunks = 0; q.n_wtiles = 0;
    if (w.planes == 3) {
      // Three planes per operand (24 mantissa bits), six of the nine plane products (the rest are below 2^-24).  The
      // tensor pipe's fp32 accumulation TRUNCATES once per instruction (tools/acc_probe.py), at the magnitude of the
      // running sum: the small products go first, onto a small accumulator, and hi x hi comes last in a sweep of its own
      // (tests/emulate_tc_accumulate.py: z error 1.1e-6 in this order, 1.6e-5 with hi x hi first).
      static const int sweeps[4][3] = {{2, 0, -1}, {1, 1, 0}, {0, 2, 1}, {0, 0, -1}};   // {A plane, W plane, W plane | -1}
      if (4 * nc > kMaxAChunks) return false;
      for (int sIdx = 0; sIdx < 4; ++sIdx)
        for (int c = 0; c < nc; ++c) {
          const int i = q.n_achunks++;
          q.a_coff[i] = sweeps[sIdx][0] * x_part_stride + c * KC;
          q.n_wpass[i] = sweeps[sIdx][2] >= 0 ? 2 : 1;
          q.w_coff[i][0] = sweeps[sIdx][1] * w.Cin + c * KC;
          q.w_coff[i][1] = (sweeps[sIdx][2] >= 0 ? sweeps[sIdx][2] : 0) * w.Cin + c * KC;
          q.n_wtiles += q.n_wpass[i] * w.ktaps;
        }
    } else {
      if (a_planes * nc > kMaxAChunks) return false;
      for (int part = 0; part < a_planes; ++part)       // x3: hi chunks meet W_hi and W_lo, lo chunks meet W_hi
        for (int c = 0; c < nc; ++c) {
          const int i = q.n_achunks++;
          q.a_coff[i] = part * x_part_stride + c * KC;
          q.n_wpass[i] = (w.x3 && part == 0) ? 2 : 1;       // (wsplit: the single activation plane meets W_hi and W_lo)
          q.w_coff[i][0] = c * KC;
          q.w_coff[i][1] = w.Cin + c * KC;
          q.n_wtiles += q.n_wpass[i] * w.ktaps;
        }
    }
    q.n_parts = n_parts; q.part_coff = part_stride;
    q.Cout = w.Cout; q.n_tile = NT; q.n_ntiles = w.Cout / NT; q.CoutT = w.CoutT;
    q.halo_mode = (halo_ok && (w.ktaps > 1 || mb > 1)) ? 1 : 0;
    const int rows = q.halo_mode ? 128 * mb + halo : 128;
    q.a_n_boxes = (rows + 255) / 256;
    q.a_box_rows = (((rows + q.a_n_boxes - 1) / q.a_n_boxes) + 7) & ~7;
    q.a_box_bytes = (uint32_t)q.a_box_rows * KC * 2;
    q.a_stage_bytes = ((uint32_t)q.a_n_boxes * q.a_box_bytes + 1023u) & ~1023u;
    q.w_box_bytes = (uint32_t)NT * KC * 2;
    q.w_stage_bytes = (q.w_box_bytes + 1023u) & ~1023u;
    q.cw = cw; q.n_echunks = NT / cw;
    q.e_box_rows = std::min(128 * mb, 256);
    q.e_n_boxes = 128 * mb / q.e_box_rows;
    q.e_part_bytes = (uint32_t)((128 * mb * cw * 2 + 1023) & ~1023);
    q.e_buf_bytes = (uint32_t)n_parts * q.e_part_bytes;
    q.n_add_bufs = 2 + (small && cw <= 32 && mb <= 2 ? 1 : 0);
    q.epi_sets = 1;
    const size_t e_bytes = ((size_t)n_adds * q.n_add_bufs + (size_t)n_outs * 2) * q.e_buf_bytes;
    const size_t w_total = (size_t)q.n_wtiles * q.w_stage_bytes;
    const int a_per_tile = q.halo_mode ? q.n_achunks : q.n_wtiles;
    size_t w_bytes;
    q.w_resident = (opt.w_resident && force_resident != 0 && q.n_ntiles == 1 && w_total <= 112 * 1024 &&
                    w_total + e_bytes + 2 * (size_t)q.a_stage_bytes <= budget) ? 1 : 0;
    if (q.w_resident) {
      w_bytes = w_total;
      q.stages_w = 1;
      q.stages_a = (int)std::min<size_t>(tc::kMaxStages, (budget - w_bytes - e_bytes) / q.a_stage_bytes);
      q.stages_a = std::min(q.stages_a, std::max(mb >= 2 ? 3 : 4, 3 * a_per_tile));
    } else if (q.halo_mode) {
      // One A stage feeds (passes x taps x mb x KC/16) MMAs; a TMA round trip is ~3000 cycles, so a short-kernel conv
      // (k = 3: ~1500 cycles of MMA per stage at C = 256) needs 3-4 stages in flight where k = 11 is fine with 2.
      const double mma_cyc = std::max(40.0, NT / 2.0);
      const double stage_cyc = (double)(w.planes > 1 ? 1.5 : 1.0) * w.ktaps * mb * (KC / 16) * mma_cyc;
      int want_a = std::min(4, std::max(2, (int)(3000.0 / stage_cyc) + 2));
      if (2 * (size_t)q.a_stage_bytes + e_bytes + 2 * (size_t)q.w_stage_bytes > budget) return false;
      while (want_a > 2 && (size_t)want_a * q.a_stage_bytes + e_bytes + 3 * (size_t)q.w_stage_bytes > budget) --want_a;
      q.stages_a = want_a;
      q.stages_w = (int)std::min<size_t>(tc::kMaxStages, (budget - e_bytes - (size_t)want_a * q.a_stage_bytes) / q.w_stage_bytes);
      if (q.stages_w < 2) { q.stages_a = 2; q.stages_w = (int)((budget - e_bytes - 2 * (size_t)q.a_stage_bytes) / q.w_stage_bytes); }
      q.stages_w = std::min(q.stages_w, tc::kMaxStages);
      w_bytes = (size_t)q.stages_w * q.w_stage_bytes;
    } else {
      const size_t per = (size_t)q.a_stage_bytes + q.w_stage_bytes;
      if (e_bytes + 2 * per > budget) return false;
      q.stages_a = q.stages_w = (int)std::min<size_t>(tc::kMaxStages, (budget - e_bytes) / per);
      w_bytes = (size_t)q.stages_w * q.w_stage_bytes;
    }
    if (q.stages_a < 2) return false;
    q.w_off = (uint32_t)(q.stages_a * q.a_stage_bytes);
    q.e_off = q.w_off + (uint32_t)w_bytes;
    q.bar_off = q.e_off + (uint32_t)e_bytes;
    *out = q;
    return true;
  };
  // Candidate plans: (blocks per tile) x (one or two CTAs per SM) x (epilogue chunk width), ranked by a small cycle
  // model of one 128-row block (constants measured on B200, tools/mma_bench.cu and the ncu source pages):
  //   MMA         the tensor pipe needs max(40, N/2) cycles per M=128 x N x 16 MMA (tools/mma_bench2.cu); the converged
  //               issue loop keeps up with it;
  //   epilogue    per chunk: ~400 cycles of CTA-wide synchronisation + TMA issue (shared by the mb blocks of the tile)
  //               plus ~150 + 4*cw cycles per block, scaled by the number of TMA-loaded / TMA-stored tensors;
  //   weights     streamed weight tiles cost their bytes / ~32 B per cycle per tile (shared by mb blocks) and want >= 3
  //               stages in flight; resident weights are free after the prologue.
  // Two CTAs per SM overlap all of it ~1.9x.
  bool planned = false;
  double best_cost = 1e30;
  TCOptions topt = opt;
  if (!opt.force_mb && !opt.force_cw && opt.force_two < 0 && opt.force_resident < 0) {
    // measured best plans (tools/tune_plans.py on a B200) take precedence over the model
    for (const TunedPlan& t : kTunedPlans)
      if (t.cin == w.Cin && t.cout == w.Cout && t.k == w.ktaps && t.n_adds == n_adds && t.n_outs == n_outs &&
          w.planes <= 2 && t.x3 == (w.x3 ? 1 : 0) && (Lq >= 128 * t.mb)) {
        topt.force_mb = t.mb; topt.force_cw = t.cw; topt.force_two = t.two; topt.force_resident = t.resident;
        break;
      }
  }
  const int mb_max = opt.max_mb;
  const double n_mma = (double)(w.planes == 3 ? 6 : w.x3 ? 3 : 1) * (w.Cin / 16) * w.ktaps;
  // N = 256 streams 32 KB of weights per (chunk, tap) for only 4 MMAs: with short kernels (k = 3) the L2 -> SM weight
  // traffic, not the tensor pipe, is the limit (ncu: 4.8 TB/s of L2 reads at C = 256, k = 3).  Splitting N into
  // 2 x 128 lets a tile take two 128-row blocks (TMEM: 2 x 2 x 128 columns), which quarters the weight bytes per row.
  int nt_cand[2] = {NT, 0};
  if (NT == 256 && opt.max_mb >= 2 && opt.split_n) nt_cand[1] = 128;
  const int nt_final_default = NT;
  for (int ci = 0; ci < 2; ++ci) {
    if (!nt_cand[ci]) continue;
    NT = nt_cand[ci];
    small = NT <= 64 && (NT <= 32 || NT % 32 == 0);
    cw_max = small ? std::min(NT, 32) : pick_cw(NT);
    if (w.planes == 3) cw_max = std::min(cw_max, 32);
  for (int two = small ? 1 : 0; two >= 0; --two)
    for (int mb = std::min(NT <= 128 ? (small ? 4 : 2) : 1, mb_max); mb >= 1; mb >>= 1)
      for (int cw = cw_max; cw >= 16; cw >>= 1) {
        if (two && 2 * mb * NT > 256) continue;   // two CTAs per SM: half the TMEM (and half the smem) each
        if ((topt.force_mb && mb != topt.force_mb) || (topt.force_cw && cw != topt.force_cw) ||
            (topt.force_two >= 0 && two != topt.force_two)) continue;
        ConvTC q;
        if (!plan(mb, cw, two ? half_budget : kSmemBudget, topt.force_resident, &q)) continue;
        if (topt.force_resident >= 0 && q.w_resident != topt.force_resident) continue;
        const double mma = n_mma * std::max(40.0, NT / 2.0);
        const double epi = (double)(NT / cw) * (400.0 / mb + 150.0 + 4.0 * cw) * (1.0 + 0.5 * n_adds + 0.5 * (n_outs - 1));
        double wcy = 0.0;
        if (!q.w_resident) {
          wcy = (double)q.n_wtiles * q.w_box_bytes / mb / 20.0;    // ~20 B / cycle / SM of streamed weights (measured)
          if (q.stages_w < 3) wcy *= 1.5;
        }
        const double stage_pen = q.stages_a < 3 && q.w_resident ? 1.1 : 1.0;   // shallow A ring exposes TMA latency
        // cost per output column so that different N tiles compare; every n-tile re-reads the activations
        const double cost = std::max(std::max(mma, epi), wcy) * stage_pen / (two ? 1.9 : 1.0) / NT * (1.0 + 0.03 * (w.Cout / NT - 1));
        if (cost < best_cost) { best_cost = cost; p = q; planned = true; }
      }
  }
  NT = planned ? p.n_tile : nt_final_default;
  small = NT <= 64 && (NT <= 32 || NT % 32 == 0);
  cw_max = small ? std::min(NT, 32) : pick_cw(NT);
  if (w.planes == 3) cw_max = std::min(cw_max, 32);
  if (!planned && (topt.force_mb || topt.force_cw)) {   // a tuned entry that does not fit this launch: use the model
    topt = TCOptions();
    topt.halo_mode = opt.halo_mode; topt.w_resident = opt.w_resident; topt.max_mb = opt.max_mb;
    for (int two = small ? 1 : 0; two >= 0 && !planned; --two)
      for (int mb = std::min(NT <= 128 ? (small ? 4 : 2) : 1, mb_max); mb >= 1 && !planned; mb >>= 1)
        for (int cw = cw_max; cw >= 16 && !planned; cw >>= 1) {
          if (two && 2 * mb * NT > 256) continue;
          planned = plan(mb, cw, two ? half_budget : kSmemBudget, -1, &p);
        }
  }
  if (!planned) return fail(VSG_EUNSUPPORTED, "conv tile does not fit in shared memory");
  const int cw = p.cw;
  const int ow = pairs ? cw / 2 : cw;                                // output channels per chunk
  p.B = B; p.Lq = Lq; p.Lout = Lout;
  p.out_stride = out_stride; p.out_phase = out_phase;
  p.tile_stride = 128 * p.mb;
  p.m_tiles_per_b = (Lq + p.tile_stride - 1) / p.tile_stride;
  p.total_tiles = p.m_tiles_per_b * p.n_ntiles * B;
  p.e_swz_mask = cw >= 64 ? 7u : cw >= 32 ? 3u : 1u;
  p.e_out_swz_mask = ow >= 64 ? 7u : ow >= 32 ? 3u : ow >= 16 ? 1u : 0u;
  p.mode = e.mode; p.mask = e.mask; p.mask_ld = e.mask_ld > 0 ? e.mask_ld : Lout; p.couple_sign = e.couple_sign;
  p.has_add0 = e.add0 != nullptr; p.has_add1 = e.add1 != nullptr;
  p.has_raw = e.out_raw != nullptr; p.has_act = e.out_act != nullptr;
  p.add0_is_act = e.add0_is_act;
  const size_t smem = 1024 + (size_t)p.bar_off + 8 * tc::kNumBars + 64;
  if (smem > kSmemMax) return fail(VSG_EUNSUPPORTED, "conv tile does not fit in shared memory (%zu B)", smem);
  p.tmem_cols = 32;
  while (p.tmem_cols < (uint32_t)(2 * p.mb * NT)) p.tmem_cols <<= 1;
  p.swizzle_code = KC == 64 ? 2u : KC == 32 ? 4u : 6u;
  p.sbo_bytes = 8u * KC * 2u;
  p.bias = e.bias; p.bcond = e.bcond; p.bcond_bs = e.bcond_bs;
  p.scale = e.scale; p.slope = e.slope;
  p.out_f32 = e.out_f32;
  p.tanh_cols = e.tanh_cols;
  p.tanh_ld = e.tanh_ld; p.tanh_s0 = e.tanh_s0; p.tanh_s1 = e.tanh_s1;
  p.mag_ch = e.mag_ch;
  p.error_flag = error_flag;

  static const bool debug_plan = getenv("VSG_DEBUG_PLAN") != nullptr;
  if (debug_plan || opt.plan_only) {
    const bool two_ctas = small && 2 * (smem + 1024) <= 228 * 1024 && 2 * p.tmem_cols <= 512;
    fprintf(stderr, "[vsg plan] conv %d->%d k%d d%d%s B%d Lq%d adds%d outs%d | %s%s mb%d cw%d halo%d resident%d stagesA%d "
                    "stagesW%d addbufs%d smem %zu KB tmem %u tiles %d\n", w.Cin, w.Cout, w.ktaps, dil, w.x3 ? " x3" : "", B, Lq,
            n_adds, n_outs, small ? "small" : "large", two_ctas ? " 2cta" : "", p.mb, p.cw, p.halo_mode, p.w_resident,
            p.stages_a, p.stages_w, p.n_add_bufs, smem / 1024, p.tmem_cols, p.total_tiles);
  }
  if (opt.plan_only) return VSG_OK;

  CUtensorMap tmA, tmAdd0, tmAdd1, tmRaw, tmAct;
  VSG_TRY(encode_3d(&tmA, x, (uint64_t)((a_planes - 1) * x_part_stride + w.Cin), (uint64_t)Lin, (uint64_t)B, (uint64_t)x_ld,
                    (uint64_t)Lin * x_ld, (uint32_t)KC, (uint32_t)p.a_box_rows, KC));
  // epilogue tensors: rows are the q positions of this (poly)phase: row stride out_stride*ld, base shifted by phase
  auto emap = [&](CUtensorMap* m, const __nv_bfloat16* base, int width, int box_c) -> int {
    return encode_3d(m, base + (size_t)out_phase * ld, (uint64_t)width, (uint64_t)Lq, (uint64_t)B,
                     (uint64_t)out_stride * ld, (uint64_t)Lout * ld, (uint32_t)box_c, (uint32_t)p.e_box_rows, box_c);
  };
  CUtensorMap tmW = w.tmap;
  if (p.n_tile != pick_ntile(w.Cout))    // the packed map's box is pick_ntile rows: rebuild it for the chosen N tile
    VSG_TRY(encode_2d(&tmW, w.w, (uint64_t)w.CinT, (uint64_t)w.ktaps * w.Cout, (uint32_t)KC, (uint32_t)p.n_tile, KC));
  tmAdd0 = tmAdd1 = tmRaw = tmAct = tmA;
  const int add_w = (n_parts - 1) * part_stride + w.Cout, out_w = (n_parts - 1) * part_stride + cout_eff;
  if (e.add0) VSG_TRY(emap(&tmAdd0, e.add0, add_w, p.cw));
  if (e.add1) VSG_TRY(emap(&tmAdd1, e.add1, add_w, p.cw));
  if (e.out_raw) VSG_TRY(emap(&tmRaw, e.out_raw, out_w, ow));
  if (e.out_act) VSG_TRY(emap(&tmAct, e.out_act, out_w, ow));
  using KernelFn = void (*)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, ConvTC);
  static const KernelFn kernels[2][EPI_SIG_COUNT] = {
      {conv_tc_kernel<false, EPI_SIG_GENERIC>, conv_tc_kernel<false, EPI_SIG_ACT>, conv_tc_kernel<false, EPI_SIG_RES_ACT>,
       conv_tc_kernel<false, EPI_SIG_LINEAR>, conv_tc_kernel<false, EPI_SIG_X6>, conv_tc_kernel<false, EPI_SIG_SUM0>,
       conv_tc_kernel<false, EPI_SIG_SUM1>, conv_tc_kernel<false, EPI_SIG_FINAL>, conv_tc_kernel<false, EPI_SIG_POST>,
       conv_tc_kernel<false, EPI_SIG_ACT_X3>, conv_tc_kernel<false, EPI_SIG_RES_ACT_X3>, conv_tc_kernel<false, EPI_SIG_SUM0_X3>,
       conv_tc_kernel<false, EPI_SIG_SUM1_X3>, conv_tc_kernel<false, EPI_SIG_FINAL_X3>, conv_tc_kernel<false, EPI_SIG_MAG>},
      {conv_tc_kernel<true, EPI_SIG_GENERIC>, conv_tc_kernel<true, EPI_SIG_ACT>, conv_tc_kernel<true, EPI_SIG_RES_ACT>,
       conv_tc_kernel<true, EPI_SIG_LINEAR>, conv_tc_kernel<true, EPI_SIG_X6>, conv_tc_kernel<true, EPI_SIG_SUM0>,
       conv_tc_kernel<true, EPI_SIG_SUM1>, conv_tc_kernel<true, EPI_SIG_FINAL>, conv_tc_kernel<true, EPI_SIG_POST>,
       conv_tc_kernel<true, EPI_SIG_ACT_X3>, conv_tc_kernel<true, EPI_SIG_RES_ACT_X3>, conv_tc_kernel<true, EPI_SIG_SUM0_X3>,
       conv_tc_kernel<true, EPI_SIG_SUM1_X3>, conv_tc_kernel<true, EPI_SIG_FINAL_X3>, conv_tc_kernel<true, EPI_SIG_MAG>}};
  // the opt-in to > 48 KB of dynamic shared memory is a per-device function attribute
  static bool attr_set_dev[64] = {false};
  bool& attr_set = attr_set_dev[P->device & 63];
  if (!attr_set) {
    for (int a = 0; a < 2; ++a)
      for (int b = 0; b < EPI_SIG_COUNT; ++b)
        VSG_CUDA_TRY(cudaFuncSetAttribute(kernels[a][b], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemMax));
    attr_set = true;
  }
  // the decoder's two dominant epilogues run kernels specialised on their feature flags (conv_tc.cuh, EPI_SIG_*)
  int sig = w.planes == 3 ? EPI_SIG_X6 : EPI_SIG_GENERIC;
  if (e.mode == EPI_TC_TANH) {
    if (a_planes != 1 || p.cw != 16 || e.tanh_cols < 1 || e.tanh_cols > 4 || !e.out_f32 || out_stride != 1 || Lq != Lout)
      return fail(VSG_EINVAL, "tanh epilogue: needs a plain-bf16 N = 16 convolution and an fp32 output");
    sig = EPI_SIG_POST;
  }
  if (e.mode == EPI_TC_MAG) {
    if (a_planes != 1 || !e.out_raw || e.out_act || e.add0 || e.add1 || e.bias || e.bcond || e.out_f32)
      return fail(VSG_EINVAL, "magnitude epilogue: needs a plain-bf16 convolution with one raw output and no bias or adds");
    sig = EPI_SIG_MAG;
  }
  if (opt.epi_sigs >= 2 && e.mode == EPI_TC_LINEAR && a_planes == 2 && e.bias && !e.bcond && !e.mask && !e.out_f32) {
    // the bf16x3 decoder's epilogues (single activated stream), as for one plane below
    if (!e.out_raw && e.out_act && !e.add1 && e.scale == 1.0f) {
      if (!e.add0) sig = EPI_SIG_ACT_X3;
      else if (e.add0_is_act) sig = EPI_SIG_RES_ACT_X3;
    } else if (e.add0 && e.add0_is_act) {
      if (e.out_raw && !e.out_act && e.scale == 1.0f) sig = e.add1 ? EPI_SIG_SUM1_X3 : EPI_SIG_SUM0_X3;
      else if (!e.out_raw && e.out_act && e.add1) sig = EPI_SIG_FINAL_X3;
    }
  }
  if (opt.epi_sigs && e.mode == EPI_TC_LINEAR && a_planes == 1 && e.bias && !e.bcond && !e.mask && !e.out_f32) {
    sig = EPI_SIG_LINEAR;
    if (!e.out_raw && e.out_act && !e.add1 && e.scale == 1.0f) {
      if (!e.add0) sig = EPI_SIG_ACT;
      else if (e.add0_is_act) sig = EPI_SIG_RES_ACT;
    } else if (opt.epi_sigs >= 2 && e.add0 && e.add0_is_act) {     // last conv2 of a resblock (single activated stream)
      if (e.out_raw && !e.out_act && e.scale == 1.0f) sig = e.add1 ? EPI_SIG_SUM1 : EPI_SIG_SUM0;
      else if (!e.out_raw && e.out_act && e.add1) sig = EPI_SIG_FINAL;
    }
  }
  // Programmatic dependent launch: the kernel's prologue (barrier init, TMEM allocation, resident-weight fetch) may
  // overlap the tail of the previous kernel in the stream; it executes griddepcontrol.wait before touching activations.
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.blockDim = dim3(tc::kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cfg.attrs = attr;
  cfg.numAttrs = opt.use_pdl ? 1 : 0;
  cudaError_t le;
  if (small) {
    // two CTAs per SM when two copies of the shared-memory carve-up (+1 KB reserved each) and of the TMEM fit
    const bool two = 2 * (smem + 1024) <= 228 * 1024 && 2 * p.tmem_cols <= 512;
    cfg.gridDim = dim3(std::min(p.total_tiles, (two ? 2 : 1) * P->sm_count));
    le = cudaLaunchKernelEx(&cfg, kernels[1][sig], tmA, tmW, tmAdd0, tmAdd1, tmRaw, tmAct, p);
  } else {
    cfg.gridDim = dim3(std::min(p.total_tiles, P->sm_count));
    le = cudaLaunchKernelEx(&cfg, kernels[0][sig], tmA, tmW, tmAdd0, tmAdd1, tmRaw, tmAct, p);
  }
  if (le != cudaSuccess) return fail(VSG_ECUDA, "launch of conv_tc_kernel failed: %s", cudaGetErrorString(le));
  VSG_LAUNCH_CHECK("conv_tc_kernel");
  static_assert(EPI_SIG_COUNT <= kImageSlots, "one launch counter per epilogue image");
  ++g_image_launches[sig];
  if (image_out) *image_out = sig;
  return VSG_OK;
}

// ---- fused ResBlock1 pair (pair_tc.cuh) ---------------------------------------------------------------------------
// 128-row blocks per tile of the fused pair: tiles of the same byte size at both channel counts (per-tile costs are what
// the low-channel stages are bound by)
static inline int pair_mb(int C) { return C == 16 ? 4 : 2; }
// TMA store boxes per tile (one box holds <= 256 rows) and valid output rows per tile.  With two boxes the box height must
// be a multiple of 8 rows so that both start on a swizzle-atom boundary of the staging tile (a few more halo rows are
// recomputed).
static inline int pair_eboxes(int C) { return (128 * pair_mb(C) + 255) / 256; }
static inline int pair_valid_rows(int C, int k) {
  const int rows = 128 * pair_mb(C) - (k - 1), n = pair_eboxes(C);
  return n == 1 ? rows : (rows / (8 * n)) * (8 * n);
}

bool pair_supported(const ConvWTC& w1, const ConvWTC& w2, int d1, int L, int n_adds, int n_outs) {
  const int C = w1.Cin, k = w1.ktaps;
  if (!w1.has_tmap || !w2.has_tmap || w1.x3 || w2.x3) return false;
  if (w1.Cout != C || w2.Cin != C || w2.Cout != C || w2.ktaps != k || (C != 16 && C != 32) || k % 2 == 0) return false;
  const int rows_t = 128 * pair_mb(C);          // rows per tile: 512 at C = 16, 256 at C = 32 (same bytes per tile)
  if ((k - 1) * d1 > 256 || L < rows_t) return false;
  // shared-memory footprint (mirrors launch_pair_tc): 2 input stages + both weight sets + 2 intermediate tiles + staging
  auto r1k = [](size_t v) { return (v + 1023) & ~(size_t)1023; };
  const int rows1 = rows_t + (k - 1) * d1, nb = (rows1 + 255) / 256, box = (((rows1 + nb - 1) / nb) + 7) & ~7;
  const size_t a1 = r1k((size_t)nb * box * C * 2), wb = (size_t)k * r1k((size_t)C * C * 2);
  const size_t tb = r1k((size_t)((rows_t + k - 1 + 7) & ~7) * C * 2), eb = (size_t)(n_adds * 2 + n_outs * 2) * r1k(rows_t * C * 2);
  return 2 * a1 + 2 * wb + 2 * tb + eb <= kSmemBudget;
}

// x_new = conv2(leaky_relu(conv1(xa) + b1)) + b2 [+ add0 + add1] [* scale]; xa = leaky_relu(x) [B, L, C] bf16.
int launch_pair_tc(const VsgPack* P, const ConvWTC& w1, const ConvWTC& w2, const __nv_bfloat16* xa, int B, int L, int d1,
                   const EpiTC& e, const TCOptions& opt, int* error_flag, cudaStream_t st, int* image_out = nullptr) {
  const int C = w1.Cin, k = w1.ktaps, mb = pair_mb(C);
  const int h2 = (k - 1) / 2, pad1 = (k - 1) * d1 / 2, halo1 = (k - 1) * d1;
  // the input is read with a halo that other CTAs' output tiles cover: an aliased output is a data race
  if ((const void*)xa == (const void*)e.out_act || (const void*)xa == (const void*)e.out_raw)
    return fail(VSG_EINVAL, "fused pair must not run in place (output aliases the activated input)");
  const int n_eboxes = pair_eboxes(C), V = pair_valid_rows(C, k);
  const int n_adds = (e.add0 ? 1 : 0) + (e.add1 ? 1 : 0), n_outs = (e.out_raw ? 1 : 0) + (e.out_act ? 1 : 0);
  ConvTC p1, p2;
  memset(&p1, 0, sizeof(p1));
  memset(&p2, 0, sizeof(p2));
  for (ConvTC* q : {&p1, &p2}) {
    q->B = B; q->Lq = L; q->Lout = L; q->KC = C; q->ktaps = k; q->n_achunks = 1; q->a_coff[0] = 0; q->n_wpass[0] = 1;
    q->w_coff[0][0] = 0; q->n_wtiles = k; q->Cout = C; q->n_tile = C; q->n_ntiles = 1; q->CoutT = C; q->out_stride = 1;
    q->mb = mb; q->tile_stride = V; q->m_tiles_per_b = (L + V - 1) / V; q->total_tiles = q->m_tiles_per_b * B;
    q->halo_mode = 1; q->w_resident = 1; q->stages_w = 1; q->n_parts = 1; q->part_coff = C;
    q->w_box_bytes = (uint32_t)C * C * 2; q->w_stage_bytes = (q->w_box_bytes + 1023u) & ~1023u;
    q->swizzle_code = C == 32 ? 4u : 6u; q->sbo_bytes = 8u * C * 2u; q->slope = 0.1f; q->scale = 1.f;
    q->error_flag = error_flag; q->cw = C; q->n_echunks = 1;
  }
  // front half: conv1 (dilated) over the activated input
  p1.dil = d1; p1.in_off0 = -h2 - pad1; p1.t_row_off = -h2; p1.bias = w1.bias;
  const int rows1 = 128 * mb + halo1;
  p1.a_n_boxes = (rows1 + 255) / 256;
  p1.a_box_rows = (((rows1 + p1.a_n_boxes - 1) / p1.a_n_boxes) + 7) & ~7;
  p1.a_box_bytes = (uint32_t)p1.a_box_rows * C * 2;
  p1.a_stage_bytes = ((uint32_t)p1.a_n_boxes * p1.a_box_bytes + 1023u) & ~1023u;
  p1.bar_slot0 = 0; p1.tmem_col0 = 0;
  // back half: conv2 (dilation 1) over the intermediate tile + the ordinary fused epilogue
  p2.dil = 1; p2.bias = w2.bias;
  const int rows2 = (128 * mb + k - 1 + 7) & ~7;
  p2.a_stage_bytes = ((uint32_t)rows2 * C * 2 + 1023u) & ~1023u;
  p2.stages_a = 2;
  p2.bar_slot0 = tc::kNumBars; p2.tmem_col0 = 2 * mb * C;
  p2.e_box_rows = V / n_eboxes; p2.e_n_boxes = n_eboxes;
  p2.e_part_bytes = (uint32_t)((128 * mb * C * 2 + 1023) & ~1023); p2.e_buf_bytes = p2.e_part_bytes;
  p2.n_add_bufs = 2;          // raised below to as many as fit (residual loads come from HBM: ~1.5 us of latency to cover)
  p2.epi_sets = opt.epi_sets; p1.epi_sets = 1;
  p2.e_swz_mask = p2.e_out_swz_mask = C >= 32 ? 3u : 1u;
  p2.mode = EPI_TC_LINEAR; p2.scale = e.scale;
  p2.has_add0 = e.add0 != nullptr; p2.has_add1 = e.add1 != nullptr;
  p2.has_raw = e.out_raw != nullptr; p2.has_act = e.out_act != nullptr;
  p2.add0_is_act = e.add0_is_act;
  p2.out_f32 = e.out_f32;
  const size_t w_bytes = (size_t)k * p1.w_stage_bytes;
  size_t e_bytes = ((size_t)n_adds * p2.n_add_bufs + (size_t)n_outs * 2) * p2.e_buf_bytes;
  size_t fixed = 2 * w_bytes + 2 * (size_t)p2.a_stage_bytes + e_bytes;
  if (fixed + 2 * (size_t)p1.a_stage_bytes > kSmemBudget) return fail(VSG_EUNSUPPORTED, "fused pair does not fit in shared memory");
  while (n_adds > 0 && p2.n_add_bufs < tc::kMaxAddBufs &&
         fixed + (size_t)n_adds * p2.e_buf_bytes + 3 * (size_t)p1.a_stage_bytes <= kSmemBudget) {
    ++p2.n_add_bufs;
    e_bytes += (size_t)n_adds * p2.e_buf_bytes;
    fixed += (size_t)n_adds * p2.e_buf_bytes;
  }
  p1.stages_a = (int)std::min<size_t>(4, (kSmemBudget - fixed) / p1.a_stage_bytes);
  p1.a_off = 0;
  p1.w_off = (uint32_t)(p1.stages_a * p1.a_stage_bytes);
  p2.a_off = p1.w_off + (uint32_t)w_bytes;
  p2.w_off = p2.a_off + 2 * p2.a_stage_bytes;
  p2.e_off = p2.w_off + (uint32_t)w_bytes;
  p2.bar_off = p2.e_off + (uint32_t)e_bytes;
  p1.bar_off = p2.bar_off;
  const size_t smem = 1024 + (size_t)p2.bar_off + 8 * (2 * tc::kNumBars) + 64;
  if (smem > kSmemMax) return fail(VSG_EUNSUPPORTED, "fused pair does not fit in shared memory (%zu B)", smem);
  p2.tmem_cols = 32;
  while (p2.tmem_cols < (uint32_t)(4 * mb * C)) p2.tmem_cols <<= 1;
  p1.tmem_cols = p2.tmem_cols;
  static const bool debug_plan = getenv("VSG_DEBUG_PLAN") != nullptr;
  if (debug_plan || opt.plan_only)
    fprintf(stderr, "[vsg plan] PAIR %d k%d d%d B%d L%d adds%d outs%d | V%d stagesA1 %d addbufs%d smem %zu KB tmem %u tiles %d\n",
            C, k, d1, B, L, n_adds, n_outs, V, p1.stages_a, p2.n_add_bufs, smem / 1024, p2.tmem_cols, p1.total_tiles);
  if (opt.plan_only) return VSG_OK;

  CUtensorMap tmA, tmAdd0, tmAdd1, tmRaw, tmAct;
  VSG_TRY(encode_3d(&tmA, xa, (uint64_t)C, (uint64_t)L, (uint64_t)B, (uint64_t)C, (uint64_t)L * C, (uint32_t)C,
                    (uint32_t)p1.a_box_rows, C));
  auto emap = [&](CUtensorMap* m, const __nv_bfloat16* base) -> int {
    return encode_3d(m, base, (uint64_t)C, (uint64_t)L, (uint64_t)B, (uint64_t)C, (uint64_t)L * C, (uint32_t)C,
                     (uint32_t)p2.e_box_rows, C);
  };
  tmAdd0 = tmAdd1 = tmRaw = tmAct = tmA;
  if (e.add0) VSG_TRY(emap(&tmAdd0, e.add0));
  if (e.add1) VSG_TRY(emap(&tmAdd1, e.add1));
  if (e.out_raw) VSG_TRY(emap(&tmRaw, e.out_raw));
  if (e.out_act) VSG_TRY(emap(&tmAct, e.out_act));
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.gridDim = dim3(std::min(p1.total_tiles, P->sm_count));
  cfg.blockDim = dim3(tc::kPairThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cfg.attrs = attr;
  cfg.numAttrs = opt.use_pdl ? 1 : 0;
  // kernel image by channel count and epilogue signature (conv_tc.cuh, EPI_SIG_*)
  using PairFn = void (*)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, ConvTC, ConvTC);
  static const PairFn pair_kernels[2][3] = {
      {pair_tc_kernel<16, EPI_SIG_GENERIC>, pair_tc_kernel<16, EPI_SIG_RES_ACT>, pair_tc_kernel<16, EPI_SIG_LINEAR>},
      {pair_tc_kernel<32, EPI_SIG_GENERIC>, pair_tc_kernel<32, EPI_SIG_RES_ACT>, pair_tc_kernel<32, EPI_SIG_LINEAR>}};
  static bool pair_attr_set_dev[64] = {false};
  bool& pair_attr_set = pair_attr_set_dev[P->device & 63];
  if (!pair_attr_set) {
    for (int a = 0; a < 2; ++a)
      for (int b = 0; b < 3; ++b)
        VSG_CUDA_TRY(cudaFuncSetAttribute(pair_kernels[a][b], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemMax));
    pair_attr_set = true;
  }
  int pv = 0;
  if (opt.epi_sigs && !e.out_f32 && e.bias) {
    pv = 2;
    if (e.add0 && e.add0_is_act && !e.add1 && e.out_act && !e.out_raw && e.scale == 1.0f) pv = 1;
  }
  cudaError_t le = cudaLaunchKernelEx(&cfg, pair_kernels[C == 16 ? 0 : 1][pv], tmA, w1.tmap, w2.tmap, tmAdd0, tmAdd1, tmRaw, tmAct, p1, p2);
  if (le != cudaSuccess) return fail(VSG_ECUDA, "launch of pair_tc_kernel failed: %s", cudaGetErrorString(le));
  VSG_LAUNCH_CHECK("pair_tc_kernel");
  if (image_out) *image_out = pv == 1 ? EPI_SIG_RES_ACT : pv == 2 ? EPI_SIG_LINEAR : EPI_SIG_GENERIC;
  return VSG_OK;
}

// ---- whole ResBlock1 in one kernel (rb_tc.cuh) --------------------------------------------------------------------
struct RbPlan { int mb, H, V, M, G, n_groups, stages_w; uint32_t tap_bytes, w_stage_bytes, buf_bytes; size_t smem; };

bool rb_plan(const ResBlockPack& rb, int C, int L, const TCOptions& opt, RbPlan* out) {
  const int k = rb.kernel, nd = (int)rb.dilations.size();
  if ((C != 16 && C != 32 && C != 64) || k % 2 == 0 || nd < 1 || 2 * nd > kRbMaxConvs) return false;
  if ((int)rb.c1_tc.size() != nd || (int)rb.c2_tc.size() != nd) return false;
  int H = 0, reach = (k - 1) / 2;
  for (int q = 0; q < nd; ++q) {
    const ConvWTC &w1 = rb.c1_tc[q], &w2 = rb.c2_tc[q];
    if (!w1.has_tmap || !w2.has_tmap || w1.x3 || w2.x3 || w1.Cin != C || w1.Cout != C || w2.Cin != C || w2.Cout != C ||
        w1.ktaps != k || w2.ktaps != k || rb.dilations[q] < 1) return false;
    H += (k - 1) / 2 * (rb.dilations[q] + 1);
    reach = std::max(reach, (k - 1) / 2 * rb.dilations[q]);
  }
  RbPlan p;
  p.H = H;
  p.M = std::max(8, (int)(1024 / (C * 2)));                 // margins keep the tile's first row 1024-byte aligned
  while (p.M < reach) p.M *= 2;
  const int mb_cap = std::min(kRbMaxBlocks, 512 / (2 * C));  // tensor memory: accumulators + fp32 residual stream
  int mb_max = opt.rb_max_mb > 0 ? std::min(opt.rb_max_mb, mb_cap) : mb_cap;
  p.tap_bytes = (uint32_t)((C * C * 2 + 1023) & ~1023);
  p.G = std::min(k, std::max(1, (int)(24576 / p.tap_bytes)));
  p.n_groups = (k + p.G - 1) / p.G;
  p.w_stage_bytes = (uint32_t)p.G * p.tap_bytes;
  // the tallest tile that fits (with >= 2 weight stages); a short utterance takes the smallest tile that covers it
  for (int mb = mb_max; mb >= 2; mb >>= 1) {
    const int V = 128 * mb - 2 * H;
    if (V < 64) return false;
    p.mb = mb; p.V = V;
    p.buf_bytes = (uint32_t)(((size_t)(2 * p.M + 128 * mb) * C * 2 + 1023) & ~(size_t)1023);
    const size_t fixed = 2 * (size_t)p.buf_bytes + 8 * tc::kRbNumBars + 64 + 1024;
    if (fixed + 2 * (size_t)p.w_stage_bytes > kSmemMax) continue;
    p.stages_w = (int)std::min<size_t>(kRbMaxWStages, (kSmemMax - fixed) / p.w_stage_bytes);
    p.smem = fixed + (size_t)p.stages_w * p.w_stage_bytes;
    const int half = mb >> 1;
    if (half >= 2 && 128 * half - 2 * H >= 64 && 128 * half - 2 * H >= L) continue;   // a smaller tile covers the utterance
    *out = p;
    return true;
  }
  return false;
}

// One ResBlock1 (decoder.py:91-104) on a channels-last activated input xa = leaky_relu(x) [B, L, C]:
//   out = (resblock(x) [+ add1]) * scale  ->  out_raw (bf16) and / or out_act = leaky_relu(out) (bf16) [, out_f32]
int launch_rb_tc(const VsgPack* P, const ResBlockPack& rb, int C, const __nv_bfloat16* xa, int B, int L,
                 const __nv_bfloat16* add1, __nv_bfloat16* out_raw, __nv_bfloat16* out_act, float* out_f32, float scale,
                 const TCOptions& opt, int* error_flag, cudaStream_t st) {
  RbPlan pl;
  if (!rb_plan(rb, C, L, opt, &pl)) return fail(VSG_EUNSUPPORTED, "resblock shape not supported by the fused kernel");
  if ((const void*)xa == (const void*)out_raw || (const void*)xa == (const void*)out_act)
    return fail(VSG_EINVAL, "fused resblock must not run in place (tiles read halo rows of their neighbours)");
  const int nd = (int)rb.dilations.size();
  RbTC p;
  memset(&p, 0, sizeof(p));
  RbMaps maps;
  memset(&maps, 0, sizeof(maps));
  p.B = B; p.L = L; p.k = rb.kernel; p.n_convs = 2 * nd;
  for (int q = 0; q < nd; ++q) {
    p.dil[2 * q] = rb.dilations[q]; p.dil[2 * q + 1] = 1;
    p.bias[2 * q] = rb.c1_tc[q].bias; p.bias[2 * q + 1] = rb.c2_tc[q].bias;
    maps.w[2 * q] = rb.c1_tc[q].tmap; maps.w[2 * q + 1] = rb.c2_tc[q].tmap;
  }
  p.mb = pl.mb; p.H = pl.H; p.V = pl.V; p.M = pl.M;
  p.m_tiles_per_b = (L + pl.V - 1) / pl.V;
  p.total_tiles = p.m_tiles_per_b * B;
  p.G = pl.G; p.n_groups = pl.n_groups; p.stages_w = pl.stages_w;
  p.tap_bytes = pl.tap_bytes; p.w_stage_bytes = pl.w_stage_bytes; p.buf_bytes = pl.buf_bytes;
  p.p_off = 0; p.q_off = pl.buf_bytes; p.w_off = 2 * pl.buf_bytes;
  p.bar_off = p.w_off + (uint32_t)pl.stages_w * pl.w_stage_bytes;
  p.tmem_cols = 32;
  while (p.tmem_cols < (uint32_t)(2 * pl.mb * C)) p.tmem_cols <<= 1;
  p.swizzle_code = C == 64 ? 2u : C == 32 ? 4u : 6u;
  p.sbo_bytes = 8u * C * 2u;
  // epilogue sets: a power of two <= 4; the (block, chunk) units of a tile must cover every set
  p.n_sets = std::max(1, std::min(opt.rb_sets, tc::kRbMaxSets));
  while (p.n_sets & (p.n_sets - 1)) --p.n_sets;
  while (p.n_sets > 1 && p.n_sets > pl.mb * (C / 16)) p.n_sets >>= 1;
  p.n_issuers = opt.rb_issuers > 0 ? opt.rb_issuers : (C == 64 ? 1 : 2);
  p.n_issuers = std::max(1, std::min(std::min(p.n_issuers, tc::kRbMaxIssuers), pl.mb));
  while (p.n_issuers & (p.n_issuers - 1)) --p.n_issuers;
  p.add1 = add1; p.out_raw = out_raw; p.out_act = out_act; p.out_f32 = out_f32;
  p.scale = scale; p.slope = 0.1f;
  p.error_flag = error_flag;
  static const bool debug_plan = getenv("VSG_DEBUG_PLAN") != nullptr;
  if (debug_plan || opt.plan_only)
    fprintf(stderr, "[vsg plan] RESBLOCK C%d k%d pairs%d B%d L%d | mb%d H%d V%d M%d G%d groups%d stagesW%d sets%d smem %zu KB "
                    "issuers%d tmem %u tiles %d\n", C, rb.kernel, nd, B, L, pl.mb, pl.H, pl.V, pl.M, pl.G, pl.n_groups, pl.stages_w,
            p.n_sets, pl.smem / 1024, p.n_issuers, p.tmem_cols, p.total_tiles);
  if (opt.plan_only) return VSG_OK;
  CUtensorMap tmA;
  const int R = 128 * pl.mb;
  VSG_TRY(encode_3d(&tmA, xa, (uint64_t)C, (uint64_t)L, (uint64_t)B, (uint64_t)C, (uint64_t)L * C, (uint32_t)C,
                    (uint32_t)std::min(R, 256), C));
  using RbFn = void (*)(CUtensorMap, RbMaps, RbTC);
  RbFn fn = C == 16 ? rb_tc_kernel<16> : C == 32 ? rb_tc_kernel<32> : rb_tc_kernel<64>;
  static bool rb_attr_set_dev[64] = {false};
  bool& attr_set = rb_attr_set_dev[P->device & 63];
  if (!attr_set) {
    for (RbFn f : {(RbFn)rb_tc_kernel<16>, (RbFn)rb_tc_kernel<32>, (RbFn)rb_tc_kernel<64>})
      VSG_CUDA_TRY(cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemMax));
    attr_set = true;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.gridDim = dim3(std::min(p.total_tiles, P->sm_count));
  cfg.blockDim = dim3((4 + 4 * p.n_sets + (p.n_issuers > 2 ? 2 : 0)) * 32);
  cfg.dynamicSmemBytes = pl.smem;
  cfg.stream = st;
  cfg.attrs = attr;
  cfg.numAttrs = opt.use_pdl ? 1 : 0;
  cudaError_t le = cudaLaunchKernelEx(&cfg, fn, tmA, maps, p);
  if (le != cudaSuccess) return fail(VSG_ECUDA, "launch of rb_tc_kernel failed: %s", cudaGetErrorString(le));
  VSG_LAUNCH_CHECK("rb_tc_kernel");
  return VSG_OK;
}

// ---- row-packed whole ResBlock1 (rp_tc.cuh) ------------------------------------------------------------------------
struct RpPlan {
  bool two_cta;
  int S, mb, H, V, n_k, packed_stages, tps, direct_stages, n_wst;
  uint32_t packed_mask, margin_bytes, buf_bytes;
  size_t smem;
};

// x3: the split-bf16 instantiation (two planes per activation tile, [W_hi | W_lo] ring stages streamed per block)
bool rp_plan(const ResBlockPack& rb, int C, int L, const TCOptions& opt, RpPlan* out, bool x3 = false) {
  const int k = rb.kernel, nd = (int)rb.dilations.size();
  if ((C != 16 && C != 32 && C != 64) || k % 2 == 0 || nd < 1 || 2 * nd > kRpMaxConvs) return false;
  if ((int)rb.c1_tc.size() != nd || (int)rb.c2_tc.size() != nd || (int)rb.c2_bsum.size() != nd) return false;
  if (x3 && (C == 64 || (int)rb.c1_x3.size() != nd || (int)rb.c2_x3.size() != nd)) return false;
  const std::vector<ConvWTC>&c1v = x3 ? rb.c1_x3 : rb.c1_tc, &c2v = x3 ? rb.c2_x3 : rb.c2_tc;
  const std::vector<ConvWTC>&c1p = x3 ? rb.c1_rp_x3 : rb.c1_rp, &c2p = x3 ? rb.c2_rp_x3 : rb.c2_rp;
  RpPlan p;
  p.S = 64 / C;
  if (L % p.S) return false;
  const int cen = (k - 1) / 2;
  int H = 0, dmax = 1;
  p.packed_mask = 0;
  for (int q = 0; q < nd; ++q) {
    const ConvWTC &w1 = c1v[q], &w2 = c2v[q];
    if (!w1.has_tmap || !w2.has_tmap || w1.x3 != x3 || w2.x3 != x3 || w1.Cin != C || w1.Cout != C || w2.Cin != C || w2.Cout != C ||
        w1.ktaps != k || w2.ktaps != k || rb.dilations[q] < 1) return false;
    H += cen * (rb.dilations[q] + 1);
    dmax = std::max(dmax, rb.dilations[q]);
    if (opt.rp_packed && p.S > 1) {
      if (rb.dilations[q] == 1 && (int)c1p.size() == nd && c1p[q].has_tmap) p.packed_mask |= 1u << (2 * q);
      if ((int)c2p.size() == nd && c2p[q].has_tmap) p.packed_mask |= 1u << (2 * q + 1);
    }
  }
  p.H = (H + p.S - 1) / p.S * p.S;
  p.n_k = (k + p.S - 1) * (C / 16);
  p.packed_stages = (p.n_k + 3) / 4;
  const uint32_t slot_bytes = std::max(1024, C * C * 2);
  p.tps = (int)(kRpStageBytes / slot_bytes);
  p.direct_stages = (k + p.tps - 1) / p.tps;
  const int reach_bytes = cen * dmax * C * 2 + 128;
  p.margin_bytes = (uint32_t)((reach_bytes + 1023) & ~1023);
  int need = 0;
  for (int c = 0; c < 2 * nd; ++c) need = std::max(need, ((p.packed_mask >> c) & 1u) ? p.packed_stages : p.direct_stages);
  // (x3: the epilogue's register budget is sized for <= 2 column chunks per thread, i.e. tiles of <= 2 blocks)
  const bool two_cta = opt.rp_two_cta && !x3 && C <= 32;
  const bool stream = x3 || two_cta;
  const size_t smem_max = two_cta ? (kSmemMax - 2048) / 2 : kSmemMax;
  const int mb_cap = stream ? 2 : kRpMaxBlocks;
  const int mb_max = opt.rp_max_mb > 0 ? std::min(opt.rp_max_mb, mb_cap) : mb_cap;
  const size_t stage_bytes = x3 ? 2 * kRpStageBytes : kRpStageBytes;
  for (int mb = mb_max; mb >= 1; --mb) {
    const int V = 128 * p.S * mb - 2 * p.H;
    if (V < 32 * p.S) return false;
    p.mb = mb; p.V = V;
    p.buf_bytes = 2 * p.margin_bytes + 16384u * (uint32_t)mb;
    const size_t fixed = (x3 ? 4 : 2) * (size_t)p.buf_bytes + 8 * tc::kRpNumBars + 64 + kRpMaxConvs * 64 * sizeof(float) + 1024;
    // x3 / two CTAs stream the ring once per block (two stages are enough to run; more is prefetch depth)
    if (fixed + (size_t)(stream ? std::min(need, 2) : need) * stage_bytes > smem_max) continue;
    // a convolution's stages are released by its last block: twice the largest need keeps a whole convolution of prefetch
    p.n_wst = (int)std::min<size_t>({(size_t)kRpMaxWStages, (size_t)2 * need, (smem_max - fixed) / stage_bytes});
    p.smem = fixed + (size_t)p.n_wst * stage_bytes;
    if (mb > 1 && 128 * p.S * (mb - 1) - 2 * p.H >= L) continue;   // a smaller tile covers the utterance
    p.two_cta = two_cta;
    *out = p;
    return true;
  }
  return false;
}

// One ResBlock1 (decoder.py:91-104) on a channels-last activated input xa = leaky_relu(x) [B, L, C]:
//   out = (resblock(x) [+ add1]) * scale  ->  out_raw (bf16) and / or out_act = leaky_relu(out) (bf16) [, out_f32]
int launch_rp_tc(const VsgPack* P, const ResBlockPack& rb, int C, const __nv_bfloat16* xa, int B, int L,
                 const __nv_bfloat16* add1, __nv_bfloat16* out_raw, __nv_bfloat16* out_act, float* out_f32, float scale,
                 const TCOptions& opt, int* error_flag, cudaStream_t st, bool x3 = false) {
  // x3: xa / add1 / out_raw are PLANAR two-plane tensors [2][B, L, C] (hi plane, then lo plane); out_act has the decoder's
  // rows [B, L, 2 C] = [hi (C) | lo (C)] per time step; out_f32 stays [B, L, C]
  RpPlan pl;
  if (!rp_plan(rb, C, L, opt, &pl, x3)) return fail(VSG_EUNSUPPORTED, "resblock shape not supported by the row-packed kernel");
  if ((const void*)xa == (const void*)out_raw || (const void*)xa == (const void*)out_act)
    return fail(VSG_EINVAL, "fused resblock must not run in place (tiles read halo rows of their neighbours)");
  const int nd = (int)rb.dilations.size();
  RpTC p;
  memset(&p, 0, sizeof(p));
  RpMaps maps;
  memset(&maps, 0, sizeof(maps));
  p.B = B; p.L = L; p.k = rb.kernel; p.n_convs = 2 * nd;
  for (int q = 0; q < nd; ++q) {
    p.dil[2 * q] = rb.dilations[q]; p.dil[2 * q + 1] = 1;
    p.bias[2 * q] = rb.c1_tc[q].bias; p.bias[2 * q + 1] = rb.c2_bsum[q];
    if (x3) {
      maps.w[2 * q] = ((pl.packed_mask >> (2 * q)) & 1u) ? rb.c1_rp_x3[q].tmap : rb.c1_x3[q].tmap;
      maps.w[2 * q + 1] = ((pl.packed_mask >> (2 * q + 1)) & 1u) ? rb.c2_rp_x3[q].tmap : rb.c2_x3[q].tmap;
    } else {
      maps.w[2 * q] = ((pl.packed_mask >> (2 * q)) & 1u) ? rb.c1_rp[q].tmap : rb.c1_tc[q].tmap;
      maps.w[2 * q + 1] = ((pl.packed_mask >> (2 * q + 1)) & 1u) ? rb.c2_rp[q].tmap : rb.c2_tc[q].tmap;
    }
  }
  p.packed_mask = pl.packed_mask; p.n_k = pl.n_k; p.packed_stages = pl.packed_stages;
  p.tps = pl.tps; p.direct_stages = pl.direct_stages;
  p.mb = pl.mb; p.H = pl.H; p.V = pl.V;
  p.spb = pl.mb >= 3 ? (opt.rp_spb2 ? 2 : 1) : 4 / pl.mb;   // epilogue warp sets per block
  if (pl.two_cta) p.spb = 2 / pl.mb;                        // (two epilogue sets per CTA)
  // (x3, two blocks: two sets per block, the blocks drained side by side -- measured 5-8 % faster than all four sets on
  // one block after the other, VSG_RP_X3_SPB4=1, although block 1's drain is the exposed part of a convolution step)
  static const bool x3_spb4 = getenv("VSG_RP_X3_SPB4") != nullptr;   // A/B aid
  if (x3 && x3_spb4) p.spb = 4;
  p.plane_stride = (long long)B * L * C;
  p.m_tiles_per_b = (L + pl.V - 1) / pl.V;
  p.total_tiles = p.m_tiles_per_b * B;
  p.n_wst = pl.n_wst;
  p.margin_bytes = pl.margin_bytes; p.buf_bytes = pl.buf_bytes;
  p.p_off = 0; p.q_off = (x3 ? 2 : 1) * pl.buf_bytes; p.w_off = (x3 ? 4 : 2) * pl.buf_bytes;
  p.bar_off = p.w_off + (uint32_t)pl.n_wst * (x3 ? 2 : 1) * kRpStageBytes;
  p.bias_off = p.bar_off + 8 * tc::kRpNumBars + 64;
  p.tmem_cols = 32;
  while (p.tmem_cols < (uint32_t)(2 * pl.mb * 64)) p.tmem_cols <<= 1;
  p.add1 = add1; p.out_raw = out_raw; p.out_act = out_act; p.out_f32 = out_f32;
  p.scale = scale; p.slope = 0.1f;
  p.error_flag = error_flag;
  p.trace = opt.rp_trace;
  static const bool debug_plan = getenv("VSG_DEBUG_PLAN") != nullptr;
  if (debug_plan || opt.plan_only)
    fprintf(stderr, "[vsg plan] ROWPACKED RESBLOCK%s C%d k%d pairs%d B%d L%d | S%d mb%d H%d V%d packed 0x%x K slices %d (stages %d) "
                    "direct stages %d ring %d margin %u smem %zu KB tmem %u tiles %d\n", x3 ? " x3" : "", C, rb.kernel, nd, B, L, pl.S, pl.mb,
            pl.H, pl.V, pl.packed_mask, pl.n_k, pl.packed_stages, pl.direct_stages, pl.n_wst,
            pl.margin_bytes, pl.smem / 1024, p.tmem_cols, p.total_tiles);
  if (opt.plan_only) return VSG_OK;
  // the input as rows of 64 channels = S time steps: [B, L, C] == [B, L / S, 64]
  CUtensorMap tmA;
  VSG_TRY(encode_3d(&tmA, xa, 64, (uint64_t)(L / pl.S), (uint64_t)B, 64, (uint64_t)L * C, 64, 128, 64));
  maps.add1 = tmA; maps.a_lo = tmA; maps.add1_lo = tmA;
  if (add1) VSG_TRY(encode_3d(&maps.add1, add1, 64, (uint64_t)(L / pl.S), (uint64_t)B, 64, (uint64_t)L * C, 64, 128, 64));
  if (x3) {   // the lo planes
    VSG_TRY(encode_3d(&maps.a_lo, xa + p.plane_stride, 64, (uint64_t)(L / pl.S), (uint64_t)B, 64, (uint64_t)L * C, 64, 128, 64));
    maps.add1_lo = maps.a_lo;
    if (add1)
      VSG_TRY(encode_3d(&maps.add1_lo, add1 + p.plane_stride, 64, (uint64_t)(L / pl.S), (uint64_t)B, 64, (uint64_t)L * C, 64, 128, 64));
  }
  using RpFn = void (*)(CUtensorMap, RpMaps, RpTC);
  RpFn fn = x3 ? (C == 16 ? (RpFn)rp_tc_kernel<16, true> : (RpFn)rp_tc_kernel<32, true>)
               : pl.two_cta ? (C == 16 ? (RpFn)rp_tc_kernel<16, false, 2> : (RpFn)rp_tc_kernel<32, false, 2>)
               : (C == 16 ? (RpFn)rp_tc_kernel<16> : C == 32 ? (RpFn)rp_tc_kernel<32> : (RpFn)rp_tc_kernel<64>);
  static bool rp_attr_set_dev[64] = {false};
  bool& attr_set = rp_attr_set_dev[P->device & 63];
  if (!attr_set) {
    for (RpFn f : {(RpFn)rp_tc_kernel<16>, (RpFn)rp_tc_kernel<32>, (RpFn)rp_tc_kernel<64>, (RpFn)rp_tc_kernel<16, true>,
                   (RpFn)rp_tc_kernel<32, true>, (RpFn)rp_tc_kernel<16, false, 2>, (RpFn)rp_tc_kernel<32, false, 2>})
      VSG_CUDA_TRY(cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemMax));
    attr_set = true;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.gridDim = dim3(std::min(p.total_tiles, (pl.two_cta ? 2 : 1) * P->sm_count));
  cfg.blockDim = dim3(pl.two_cta ? (4 + 4 * 2) * 32 : tc::kRpThreads);
  cfg.dynamicSmemBytes = pl.smem;
  cfg.stream = st;
  cfg.attrs = attr;
  cfg.numAttrs = opt.use_pdl ? 1 : 0;
  cudaError_t le = cudaLaunchKernelEx(&cfg, fn, tmA, maps, p);
  if (le != cudaSuccess) return fail(VSG_ECUDA, "launch of rp_tc_kernel failed: %s", cudaGetErrorString(le));
  VSG_LAUNCH_CHECK("rp_tc_kernel");
  return VSG_OK;
}

size_t dec_max_elems(const VsgPack* P, int B, int T) {
  size_t m = (size_t)B * P->cfg.dec_upsample_initial_channel * T;
  long long L = T;
  for (const UpStage& st : P->ups) {
    L *= st.rate;
    m = std::max(m, (size_t)B * st.Cout * (size_t)L);
  }
  return m;
}

}  // namespace

// Conv1d-style weight W[co][ci][j] -> bf16 [j][co][ci] (K-major rows) + its 2-D TMA map.
// planes = 2 ("x3"): every row is [W_hi (Cin) | W_lo (Cin)] with W_hi = bf16(W), W_lo = bf16(W - W_hi);
// planes = 3: [W_hi | W_mid | W_lo], the fp32 weight exactly.
int pack_conv_tc(VsgPack* P, const std::vector<float>& W, const std::vector<float>& b, int Cout, int Cin, int k,
                 ConvWTC* out, int planes) {
  const int CinT = planes * Cin;
  out->Cin = Cin; out->Cout = Cout; out->CinT = CinT; out->CoutT = Cout; out->ktaps = k;
  out->has_tmap = false; out->x3 = planes == 2; out->planes = planes;
  const int KC = pick_kc(Cin), NT = pick_ntile(Cout);
  if (KC == 0 || NT == 0 || k < 1) return VSG_OK;   // not representable on the tensor-core path; fp32 mode still works
  std::vector<__nv_bfloat16> wp((size_t)k * Cout * CinT);
  for (int j = 0; j < k; ++j)
    for (int co = 0; co < Cout; ++co)
      for (int ci = 0; ci < Cin; ++ci) {
        float v = W[((size_t)co * Cin + ci) * k + j];
        for (int pl = 0; pl < planes; ++pl) {
          const __nv_bfloat16 h = __float2bfloat16(v);
          wp[((size_t)j * Cout + co) * CinT + (size_t)pl * Cin + ci] = h;
          v -= __bfloat162float(h);
        }
      }
  void* dw = nullptr;
  VSG_CUDA_TRY(cudaMalloc(&dw, wp.size() * sizeof(__nv_bfloat16) + 256));
  P->allocs.push_back(dw);
  VSG_CUDA_TRY(cudaMemcpy(dw, wp.data(), wp.size() * sizeof(__nv_bfloat16), cudaMemcpyHostToDevice));
  out->w = (__nv_bfloat16*)dw;
  void* db = nullptr;
  VSG_CUDA_TRY(cudaMalloc(&db, (size_t)Cout * sizeof(float) + 256));
  P->allocs.push_back(db);
  VSG_CUDA_TRY(cudaMemcpy(db, b.data(), (size_t)Cout * sizeof(float), cudaMemcpyHostToDevice));
  out->bias = (float*)db;
  VSG_TRY(encode_2d(&out->tmap, dw, (uint64_t)CinT, (uint64_t)k * Cout, (uint32_t)KC, (uint32_t)NT, KC));
  out->has_tmap = true;
  return VSG_OK;
}

// ConvTranspose1d(Cin -> Cout, k, stride = rate, padding = (k - rate) / 2) with weight W[ci][co][j] as convolutions over
// the input rate.  Polyphase split: y[q*s + r] = sum_{jj} sum_ci x[ci, q + in_off0 + jj] * W[ci][co][j0 + s*(n_r-1-jj)].
int pack_upsampler(VsgPack* P, const std::vector<float>& W, const std::vector<float>& b, int Cin, int Cout, int rate, int k,
                   UpStage* out, std::vector<std::vector<float>>* phase_w) {
  UpStage& st = *out;
  st.rate = rate; st.kernel = k; st.Cin = Cin; st.Cout = Cout; st.pad = (k - rate) / 2;
  if (rate < 1 || k < rate || (k - rate) % 2)
    return fail(VSG_EUNSUPPORTED, "upsampler: kernel %d / stride %d needs kernel >= stride and (kernel - stride) even", k, rate);
  st.phases.resize(st.rate);
  if (phase_w) phase_w->assign(st.rate, std::vector<float>());
  for (int r = 0; r < st.rate; ++r) {
    const int s = st.rate, p = st.pad;
    const int j0 = (r + p) % s;
    const int nr = (k - 1 - j0) / s + 1;
    const int cr = (r + p - j0) / s;
    UpsPhase& ph = st.phases[r];
    ph.in_off0 = cr - nr + 1;
    std::vector<float> Wc((size_t)st.Cout * st.Cin * nr);   // as a Conv1d weight [co][ci][jj]
    for (int co = 0; co < st.Cout; ++co)
      for (int ci = 0; ci < st.Cin; ++ci)
        for (int jj = 0; jj < nr; ++jj)
          Wc[((size_t)co * st.Cin + ci) * nr + jj] = W[((size_t)ci * st.Cout + co) * k + j0 + s * (nr - 1 - jj)];
    VSG_TRY(pack_conv_tc(P, Wc, b, st.Cout, st.Cin, nr, &ph.tc));
    VSG_TRY(pack_conv_tc(P, Wc, b, st.Cout, st.Cin, nr, &ph.x3, 2));
    if (phase_w) (*phase_w)[r] = std::move(Wc);
  }
  {   // merged polyphase convolution for the tensor-core path (one launch, contiguous stores)
    int off_min = 1 << 30, off_max = -(1 << 30);
    for (int r = 0; r < st.rate; ++r) {
      const int nr = (k - 1 - (r + st.pad) % st.rate) / st.rate + 1;
      off_min = std::min(off_min, st.phases[r].in_off0);
      off_max = std::max(off_max, st.phases[r].in_off0 + nr - 1);
    }
    const int kt = off_max - off_min + 1, s = st.rate, p = st.pad;
    std::vector<float> Wm((size_t)s * st.Cout * st.Cin * kt, 0.f), bm((size_t)s * st.Cout);
    for (int r = 0; r < s; ++r) {
      const int j0 = (r + p) % s, nr = (k - 1 - j0) / s + 1, off_r = st.phases[r].in_off0;
      for (int co = 0; co < st.Cout; ++co) {
        bm[(size_t)r * st.Cout + co] = b[co];
        for (int ci = 0; ci < st.Cin; ++ci)
          for (int t = 0; t < kt; ++t) {
            const int tp = off_min + t - off_r;            // tap index inside phase r
            if (tp < 0 || tp >= nr) continue;
            Wm[(((size_t)r * st.Cout + co) * st.Cin + ci) * kt + t] = W[((size_t)ci * st.Cout + co) * k + j0 + s * (nr - 1 - tp)];
          }
      }
    }
    st.merged_in_off0 = off_min;
    VSG_TRY(pack_conv_tc(P, Wm, bm, s * st.Cout, st.Cin, kt, &st.merged_tc));
    VSG_TRY(pack_conv_tc(P, Wm, bm, s * st.Cout, st.Cin, kt, &st.merged_x3, 2));   // (bf16x3: used where the output is planar)
  }
  return VSG_OK;
}

// Dilation-1 Conv1d(C -> C, k) in the row-packed form of rp_tc.cuh: S = 64 / C consecutive time steps are one row of 64
// channels; output column n = s' * C + co of a row is fed by the 16-wide K slices m = 0 .. (k + S - 1) * C / 16 - 1 of the
// input, slice m = channels 16 (m % KK) .. of input sub-step sigma = m / KK - (k-1)/2 (KK = C / 16), through tap
// j = sigma - s' + (k-1)/2:   W'[m][n][ci'] = W[co][16 (m % KK) + ci'][j]   (zero outside the k taps).
// Four slices share one [64 x 64] SWIZZLE_128B tile (K index = 16 (m % 4) + ci'): packed as Conv1d(64 -> 64, ceil(n_k / 4) taps).
int pack_conv_rowpacked(VsgPack* P, const std::vector<float>& W, int C, int k, ConvWTC* out, int planes) {
  out->has_tmap = false;
  if ((C != 16 && C != 32) || k % 2 == 0) return VSG_OK;
  const int S = 64 / C, KK = C / 16, cen = (k - 1) / 2, n_k = (k + S - 1) * KK, n_g = (n_k + 3) / 4;
  std::vector<float> Wp((size_t)64 * 64 * n_g, 0.f), bz(64, 0.f);
  for (int m = 0; m < n_k; ++m) {
    const int sigma = m / KK - cen, c_lo = 16 * (m % KK);
    for (int sp = 0; sp < S; ++sp) {
      const int j = sigma - sp + cen;
      if (j < 0 || j >= k) continue;
      for (int co = 0; co < C; ++co)
        for (int ci = 0; ci < 16; ++ci)
          Wp[((size_t)(sp * C + co) * 64 + 16 * (m % 4) + ci) * n_g + m / 4] = W[((size_t)co * C + c_lo + ci) * k + j];
    }
  }
  return pack_conv_tc(P, Wp, bz, 64, 64, n_g, out, planes);   // planes = 2: rows [W_hi (64) | W_lo (64)]
}

int pack_resblock_bias_sums(VsgPack* P, const std::vector<std::vector<float>>& b2, ResBlockPack* rb) {
  rb->c2_bsum.assign(b2.size(), nullptr);
  std::vector<float> acc;
  for (size_t q = 0; q < b2.size(); ++q) {
    if (q == 0) acc = b2[0];
    else for (size_t i = 0; i < acc.size() && i < b2[q].size(); ++i) acc[i] += b2[q][i];
    void* d = nullptr;
    VSG_CUDA_TRY(cudaMalloc(&d, acc.size() * sizeof(float) + 256));
    P->allocs.push_back(d);
    VSG_CUDA_TRY(cudaMemcpy(d, acc.data(), acc.size() * sizeof(float), cudaMemcpyHostToDevice));
    rb->c2_bsum[q] = (float*)d;
  }
  return VSG_OK;
}

bool x3_flow_on_tensor_cores() {
  static const bool ffma = getenv("VSG_X3_FLOW_FFMA") != nullptr && getenv("VSG_X3_FLOW_FFMA")[0] == '1';
  return !ffma;
}

size_t flow_ws_bytes_tc(const VsgPack* P, int B, int T, int planes) {
  const VsgConfig& c = P->cfg;
  size_t n = 0;
  n += align256((size_t)B * c.flow_n_flows * 2 * c.flow_hidden * c.flow_n_layers * sizeof(float));   // cond
  n += align256((size_t)B * T * c.flow_channels * 2 * planes);                                      // state, channels-last
  n += 3 * align256((size_t)B * T * c.flow_hidden * 2 * planes);                                    // h, acts, out
  return n + 512;
}

// ResidualCouplingBlock.forward (modules/visinger/flow.py:33-40) on the tensor-core kernels.  The coupling state,
// WaveNet state, gate output and skip sum all live channels-last in bf16; every elementwise op of the reference
// (mask multiplies, gate, residual / skip routing, coupling) is an epilogue of the convolution that produces it.
// planes = 1: plain bf16 (throughput mode).  planes = 3: every tensor and weight is three bf16 planes (hi, mid, lo =
// the fp32 value exactly) and every product runs as six plane products, small ones first (launch_conv_tc): the flow at
// north_star's fp32 tolerance (z <= 1e-5) on tcgen05 -- the bf16x3 precision mode.
int flow_forward_tc(const VsgPack* P, const float* x, const float* mask, const float* g, float* y, int B, int T,
                    int reverse, Workspace& ws, cudaStream_t st, int planes, const float* out_mask, const float* ps_logs, const float* ps_noise,
                    int x_ld) {
  const VsgConfig& c = P->cfg;
  const int C = c.flow_channels, H = c.flow_hidden, NL = c.flow_n_layers, NF = c.flow_n_flows, half = C / 2;
  const int K = c.flow_kernel_size;
  const bool x6 = planes == 3;
  if (planes != 1 && planes != 3) return fail(VSG_EINVAL, "flow_forward_tc: planes must be 1 or 3");
  if (!P->flow_layers.empty() && !P->flow_layers[0].pre_tc[0].has_tmap)
    return fail(VSG_EUNSUPPORTED, "bf16 flow needs channels/2 and hidden_channels to be multiples of 16");
  const int condO = 2 * H * NL;
  typedef __nv_bfloat16 bf;
  float* cond = ws.take<float>((size_t)B * NF * condO);
  bf* u = ws.take<bf>((size_t)B * T * C * planes);        // rows [hi (C) | mid (C) | lo (C)]
  // WaveNet state h and skip sum `out` side by side: rows [h (H) | out (H)] per plane, so that res_skip_layers[i] is one
  // launch (the Conv1d(H -> 2H) it is in the reference) and `pre`, zero-extended to 2H channels, also clears the skip sum
  bf* hs = ws.take<bf>((size_t)B * T * 2 * H * planes);
  bf* acts = ws.take<bf>((size_t)B * T * H * planes);
  int* err = ws.take<int>(1);
  if (ws.overflow) return fail(VSG_ENOMEM, "flow workspace too small: need %zu bytes", ws.off);
  VSG_CUDA_TRY(cudaMemsetAsync(err, 0, sizeof(int), st));
  const TCOptions opt = g_default_opts;
  const bool merged = opt.flow_merge != 0;
  bf* const h = hs;
  bf* const out = hs + H;
  const int hs_ld = planes * 2 * H;                       // row width of hs; its planes are 2H channels apart
  const int cond_bs = merged ? NF * condO : condO;        // floats between the utterances of the condition table
  if (c.flow_gin > 0) {
    if (!g) return fail(VSG_EINVAL, "flow was built with gin_channels=%d but g is NULL", c.flow_gin);
    if (merged) {   // every flow's cond_layer in one GEMV launch: cond[b][f * condO + o]
      VSG_TRY(launch_cond(P->flow_cond_w, P->flow_cond_b, g, cond, NF * condO, c.flow_gin, B, st));
    } else {
      for (int f = 0; f < NF; ++f)
        VSG_TRY(launch_cond(P->flow_layers[f].cond_w, P->flow_layers[f].cond_b, g, cond + (size_t)f * condO * B, condO,
                            c.flow_gin, B, st));
    }
  }
  {
    dim3 grid((T + 31) / 32, (C + 31) / 32, B), block(32, 8);
    transpose_to_bf16_kernel<<<grid, block, 0, st>>>(x, u, C, T, planes, ps_logs, ps_noise, mask, x_ld);   // (ps_*: x = mu_p, prior sampling fused)
    VSG_LAUNCH_CHECK("transpose_to_bf16_kernel");
  }
  for (int step = 0; step < NF; ++step) {
    const int f = reverse ? NF - 1 - step : step;
    const int flipped = reverse ? (NF - f) & 1 : f & 1;
    const FlowLayer& fl = P->flow_layers[f];
    const bf* x0 = u + (flipped ? half : 0);
    bf* x1 = u + (flipped ? 0 : half);
    {  // h = pre(x0) * mask  (merged: and out = 0)
      const ConvWTC& w = merged ? fl.pre2_tc[flipped][x6 ? 1 : 0] : x6 ? fl.pre_x6[flipped] : fl.pre_tc[flipped];
      EpiTC e;
      e.bias = w.bias; e.mask = mask; e.mask_ld = x_ld; e.out_raw = hs;
      if (!merged) { e.ld = hs_ld; e.part_stride = 2 * H; }
      VSG_TRY(launch_conv_tc(P, w, x0, B, T, 0, 1, T, 1, 0, T, e, opt, err, st, planes * C, C));
    }
    int dil = 1;
    for (int i = 0; i < NL; ++i) {
      const bool last = (i == NL - 1);
      {  // acts = tanh(.) * sigmoid(.) of in_layer(h) + cond
        const ConvWTC& w = x6 ? fl.in_x6[i] : fl.in_tc[i];
        EpiTC e;
        e.mode = EPI_TC_GATE; e.bias = w.bias; e.out_raw = acts;
        if (c.flow_gin > 0) {
          e.bcond = merged ? cond + (size_t)f * condO + (size_t)i * 2 * H : cond + (size_t)f * condO * B + (size_t)i * 2 * H;
          e.bcond_bs = cond_bs;
        }
        VSG_TRY(launch_conv_tc(P, w, h, B, T, -((K * dil - dil) / 2), dil, T, 1, 0, T, e, opt, err, st, hs_ld, 2 * H));
      }
      if (merged && !last) {  // [h | out] = ([h | out] + res_skip(acts)) * mask   (masking the running skip sum is a no-op
                              //  on the valid frames and the sum is masked after the last layer anyway, encoder.py:195)
        const ConvWTC& w = fl.rs_tc[x6 ? 1 : 0][i];
        EpiTC e;
        e.bias = w.bias; e.add0 = hs; e.mask = mask; e.mask_ld = x_ld; e.out_raw = hs;
        VSG_TRY(launch_conv_tc(P, w, acts, B, T, 0, 1, T, 1, 0, T, e, opt, err, st));
      } else {
        if (!last) {  // h = (h + res(acts)) * mask
          const ConvWTC& w = x6 ? fl.res_x6[i] : fl.res_tc[i];
          EpiTC e;
          e.bias = w.bias; e.add0 = h; e.mask = mask; e.mask_ld = x_ld; e.out_raw = h; e.ld = hs_ld; e.part_stride = 2 * H;
          VSG_TRY(launch_conv_tc(P, w, acts, B, T, 0, 1, T, 1, 0, T, e, opt, err, st));
        }
        {  // out (+)= skip(acts); masked after the last layer
          const ConvWTC& w = x6 ? fl.skip_x6[i] : fl.skip_tc[i];
          EpiTC e;
          e.bias = w.bias; e.add0 = (i > 0 || merged) ? out : nullptr; e.mask = last ? mask : nullptr; e.mask_ld = x_ld; e.out_raw = out;
          e.ld = hs_ld; e.part_stride = 2 * H;
          VSG_TRY(launch_conv_tc(P, w, acts, B, T, 0, 1, T, 1, 0, T, e, opt, err, st));
        }
      }
      dil *= c.flow_dilation_rate;
    }
    {  // m = post(out) * mask ; x1 = (x1 - m) * mask | m + x1 * mask
      const ConvWTC& w = x6 ? fl.post_x6[flipped] : fl.post_tc[flipped];
      EpiTC e;
      e.mode = EPI_TC_COUPLE; e.couple_sign = reverse ? -1 : 1;
      e.bias = w.bias; e.mask = mask; e.mask_ld = x_ld; e.add0 = x1; e.out_raw = x1; e.ld = planes * C; e.part_stride = C;
      VSG_TRY(launch_conv_tc(P, w, out, B, T, 0, 1, T, 1, 0, T, e, opt, err, st, hs_ld, 2 * H));
    }
  }
  {
    dim3 grid((T + 31) / 32, (C + 31) / 32, B), block(32, 8);
    transpose_from_bf16_kernel<<<grid, block, 0, st>>>(u, y, C, T, (NF & 1) ? 1 : 0, planes, out_mask, x_ld);   // (out_mask: y * mask)
    VSG_LAUNCH_CHECK("transpose_from_bf16_kernel");
  }
  return VSG_OK;
}

size_t posterior_ws_bytes_tc(const VsgPack* P, int B, int T) {
  const EncPack& e = P->enc;
  size_t n = 0;
  n += align256((size_t)B * 2 * e.hidden * e.n_layers * sizeof(float));          // cond
  n += align256((size_t)B * T * e.in_pad * 2);                                     // input, channels-last, padded rows
  n += 3 * align256((size_t)B * T * e.hidden * 2);                                 // h, acts, out
  n += align256((size_t)B * T * 2 * e.out_channels * 2);                           // stats, channels-last
  return n + 512;
}

// PosteriorEncoder.forward (modules/visinger/encoder.py:92-98) on the tensor-core kernels: the same WaveNet launches as
// the flow; `pre` contracts the (padded) input channels in slabs of <= 1024, chained through the residual input.
int posterior_forward_tc(const VsgPack* P, const float* x, const float* mask, const float* g, const float* noise,
                         float* z, float* stats, int B, int T, Workspace& ws, cudaStream_t st) {
  const EncPack& en = P->enc;
  __nv_bfloat16* u = ws.take<__nv_bfloat16>((size_t)B * T * en.in_pad);
  if (ws.overflow) return fail(VSG_ENOMEM, "posterior workspace too small: need %zu bytes", ws.off);
  {
    dim3 grid((T + 31) / 32, (en.in_pad + 31) / 32, B), block(32, 8);
    transpose_pad_to_bf16_kernel<<<grid, block, 0, st>>>(x, u, en.in_channels, en.in_pad, T);
    VSG_LAUNCH_CHECK("transpose_pad_to_bf16_kernel");
  }
  return posterior_core_tc(P, u, mask, g, noise, z, stats, B, T, ws, st);
}

int posterior_core_tc(const VsgPack* P, const __nv_bfloat16* u, const float* mask, const float* g, const float* noise,
                      float* z, float* stats, int B, int T, Workspace& ws, cudaStream_t st) {
  const EncPack& en = P->enc;
  const int H = en.hidden, NL = en.n_layers, K = en.kernel, CinP = en.in_pad, Co = en.out_channels;
  if (en.pre_tc.empty() || !en.pre_tc[0].has_tmap || !en.proj_tc.has_tmap || (int)en.wn.in_tc.size() != NL ||
      !en.wn.in_tc[0].has_tmap)
    return fail(VSG_EUNSUPPORTED, "bf16 posterior encoder needs hidden and 2 * out channels to be multiples of 16");
  const int condO = 2 * H * NL;
  typedef __nv_bfloat16 bf;
  float* cond = ws.take<float>((size_t)B * condO);
  bf* h = ws.take<bf>((size_t)B * T * H);
  bf* acts = ws.take<bf>((size_t)B * T * H);
  bf* out = ws.take<bf>((size_t)B * T * H);
  bf* sb = ws.take<bf>((size_t)B * T * 2 * Co);
  int* err = ws.take<int>(1);
  if (ws.overflow) return fail(VSG_ENOMEM, "posterior workspace too small: need %zu bytes", ws.off);
  VSG_CUDA_TRY(cudaMemsetAsync(err, 0, sizeof(int), st));
  const TCOptions opt = g_default_opts;
  if (en.gin > 0) {
    if (!g) return fail(VSG_EINVAL, "posterior encoder was built with gin_channels=%d but g is NULL", en.gin);
    VSG_TRY(launch_cond(en.wn.cond_w, en.wn.cond_b, g, cond, condO, en.gin, B, st));
  }
  for (size_t s = 0; s < en.pre_tc.size(); ++s) {   // h = pre(x) * mask, one launch per input-channel slab
    const bool last = (s + 1 == en.pre_tc.size());
    EpiTC e;
    e.bias = en.pre_tc[s].bias;                      // (only slab 0 carries the bias)
    e.add0 = s > 0 ? h : nullptr;
    e.mask = last ? mask : nullptr;
    e.out_raw = h;
    VSG_TRY(launch_conv_tc(P, en.pre_tc[s], u + en.pre_c0[s], B, T, 0, 1, T, 1, 0, T, e, opt, err, st, CinP));
  }
  int dil = 1;
  for (int i = 0; i < NL; ++i) {
    const bool last = (i == NL - 1);
    {
      EpiTC e;
      e.mode = EPI_TC_GATE; e.bias = en.wn.in_tc[i].bias; e.out_raw = acts;
      if (en.gin > 0) { e.bcond = cond + (size_t)i * 2 * H; e.bcond_bs = condO; }
      VSG_TRY(launch_conv_tc(P, en.wn.in_tc[i], h, B, T, -((K * dil - dil) / 2), dil, T, 1, 0, T, e, opt, err, st));
    }
    if (!last) {
      EpiTC e;
      e.bias = en.wn.res_tc[i].bias; e.add0 = h; e.mask = mask; e.out_raw = h;
      VSG_TRY(launch_conv_tc(P, en.wn.res_tc[i], acts, B, T, 0, 1, T, 1, 0, T, e, opt, err, st));
    }
    {
      EpiTC e;
      e.bias = en.wn.skip_tc[i].bias; e.add0 = (i > 0) ? out : nullptr; e.mask = last ? mask : nullptr; e.out_raw = out;
      VSG_TRY(launch_conv_tc(P, en.wn.skip_tc[i], acts, B, T, 0, 1, T, 1, 0, T, e, opt, err, st));
    }
    dil *= en.dil_rate;
  }
  {  // stats = proj(h) * mask
    EpiTC e;
    e.bias = en.proj_tc.bias; e.mask = mask; e.out_raw = sb;
    VSG_TRY(launch_conv_tc(P, en.proj_tc, out, B, T, 0, 1, T, 1, 0, T, e, opt, err, st));
  }
  {
    dim3 grid((T + 31) / 32, (2 * Co + 31) / 32, B), block(32, 8);
    transpose_from_bf16_kernel<<<grid, block, 0, st>>>(sb, stats, 2 * Co, T, 0, 1);
    VSG_LAUNCH_CHECK("transpose_from_bf16_kernel");
  }
  const long long n = (long long)B * Co * T;
  posterior_sample_from_stats_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(stats, noise, mask, z, Co, T, n);
  VSG_LAUNCH_CHECK("posterior_sample_from_stats_kernel");
  return VSG_OK;
}

// u [B, T, in_pad] = |STFT| * mask in bf16: the framed rows, then Conv1d(hopP -> 2 in_pad, taps) on tcgen05 with the
// magnitude epilogue (conv_tc.cuh, EPI_TC_MAG), which also zeroes the pad channels.
int spectrogram_tc(const VsgPack* P, const SpecPack& S, int in_pad, const float* wav, const int32_t* lengths,
                   const float* mask, __nv_bfloat16* u, int B, int T, Workspace& ws, cudaStream_t st, int t0, int T_len) {
  if (!S.tc.has_tmap || S.tc.Cout != 2 * in_pad) return fail(VSG_EUNSUPPORTED, "no tensor-core spectrogram pack");
  const int R = T + S.taps - 1;
  if (!T_len) T_len = T;
  const size_t mark = ws.off;
  __nv_bfloat16* rows = ws.take<__nv_bfloat16>((size_t)B * R * S.hopP);
  int* err = ws.take<int>(1);
  if (ws.overflow) return fail(VSG_ENOMEM, "spectrogram workspace too small: need %zu bytes", ws.off);
  VSG_CUDA_TRY(cudaMemsetAsync(err, 0, sizeof(int), st));
  const long long n = (long long)B * R * S.hopP;
  spec_frames_kernel<true><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(wav, lengths, rows, T_len, R, S.hop, S.hopP, S.off,
                                                                          S.taps, n, t0, (long long)T_len * S.hop);
  VSG_LAUNCH_CHECK("spec_frames_kernel");
  EpiTC e;
  e.mode = EPI_TC_MAG; e.mask = mask; e.out_raw = u; e.mag_ch = S.bins;
  VSG_TRY(launch_conv_tc(P, S.tc, rows, B, R, 0, 1, T, 1, 0, T, e, g_default_opts, err, st));
  ws.off = mark;   // stream-ordered: the next user of the rows runs after the convolution
  return VSG_OK;
}

int widen_bf16(const __nv_bfloat16* x, float* y, int B, int C, int ld, int T, cudaStream_t st) {
  dim3 grid((T + 31) / 32, (C + 31) / 32, B), block(32, 8);
  widen_bf16_kernel<<<grid, block, 0, st>>>(x, y, C, ld, T);
  VSG_LAUNCH_CHECK("widen_bf16_kernel");
  return VSG_OK;
}

size_t relenc_ws_bytes_tc(const VsgPack* P, int B, int T, int g_t) {
  const RelEncPack& e = P->relenc;
  size_t n = 0;
  n += align256((size_t)B * T * e.hidden * 2) * 2;            // x, attention output
  n += align256((size_t)B * T * 3 * e.hidden * 2);            // q | k | v
  n += align256((size_t)B * T * e.filter * 2);                // FFN hidden
  n += align256((size_t)B * e.hidden * (g_t ? T : 1) * sizeof(float));
  if (T > 128 * tc::kAtMaxTiles)                              // split-key attention: per-chunk partial outputs
    n += align256(attention_split_floats(B, T, e.n_heads, e.hidden / e.n_heads, tc::kAtMaxTiles) * sizeof(float));
  return n + 512;
}

namespace {
// chunk_tiles = 0: one launch over all key tiles (T <= 2048), normalised output.  chunk_tiles > 0: the split-key launch
// over key chunks of that many tiles, its partials in `part` (attention_split_floats), then the combine.
template <int DK>
int launch_attention_bf16(const __nv_bfloat16* qkv, const float* mask, const float* ek, const float* ev, __nv_bfloat16* o, int B,
                          int n_heads, int T, int w, int chunk_tiles, float* part, int* err, cudaStream_t st) {
  const int n_tiles = (T + 127) / 128;
  if (chunk_tiles == 0 && n_tiles > tc::kAtMaxTiles)
    return fail(VSG_EUNSUPPORTED, "attention: sequence of %d frames (supported: <= %d)", T, 128 * tc::kAtMaxTiles);
  if (chunk_tiles < 0 || chunk_tiles > tc::kAtMaxTiles || (chunk_tiles > 0 && !part))
    return fail(VSG_EINVAL, "attention: key chunk of %d tiles (supported: 1 .. %d, with a partials buffer)", chunk_tiles, tc::kAtMaxTiles);
  if (w > 7) return fail(VSG_EUNSUPPORTED, "attention: relative-position window %d (supported: <= 7)", w);
  const int H = n_heads * DK;
  constexpr int CW = AttnSmem<DK>::CW;
  CUtensorMap tm;   // the fused projection's output [B, T, 3H] as (channels, frames, utterances)
  VSG_TRY(encode_3d(&tm, qkv, (uint64_t)3 * H, (uint64_t)T, (uint64_t)B, (uint64_t)3 * H, (uint64_t)T * 3 * H, (uint32_t)CW, 128, CW));
  AttnTC p;
  p.B = B; p.T = T; p.n_heads = n_heads; p.w = w; p.n_tiles = n_tiles; p.chunk_tiles = chunk_tiles ? chunk_tiles : n_tiles;
  p.mask = mask; p.Ek = ek; p.Ev = ev; p.o = o; p.error_flag = err;
  const int n_chunks = (n_tiles + p.chunk_tiles - 1) / p.chunk_tiles;
  p.o_part = p.m_part = p.l_part = nullptr;
  if (chunk_tiles) {
    p.o_part = part;
    p.m_part = part + (size_t)n_chunks * B * T * H;
    p.l_part = p.m_part + (size_t)n_chunks * B * n_heads * T;
  }
  const size_t sm = AttnSmem<DK>::bytes;
  static bool attr_set[64] = {false};
  int dev = 0;
  VSG_CUDA_TRY(cudaGetDevice(&dev));
  if (!attr_set[dev & 63]) {
    // dk = 128 needs 261 536 bytes (Q, two K, two V and two P tiles), more than the 232 448 a B200 block may opt in to
    int optin = 0;
    VSG_CUDA_TRY(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    if (sm > (size_t)optin)
      return fail(VSG_EUNSUPPORTED, "attention head width %d needs %zu bytes of shared memory per block, above this device's "
                  "limit of %d (supported head widths: 16, 32, 48, 64, 96)", DK, sm, optin);
    VSG_CUDA_TRY(cudaFuncSetAttribute(relenc_attention_tc_kernel<DK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    attr_set[dev & 63] = true;
  }
  dim3 grid(n_tiles * n_chunks, n_heads, B);
  relenc_attention_tc_kernel<DK><<<grid, tc::kAtThreads, sm, st>>>(tm, p);
  VSG_LAUNCH_CHECK("relenc_attention_tc_kernel");
  if (chunk_tiles) {
    const long long n = (long long)B * T * H / 8;
    attention_combine_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(p.o_part, p.m_part, p.l_part, o, B, T, n_heads, DK,
                                                                           n_chunks);
    VSG_LAUNCH_CHECK("attention_combine_kernel");
  }
  return VSG_OK;
}

int attention_bf16(int dk, const __nv_bfloat16* qkv, const float* mask, const float* ek, const float* ev, __nv_bfloat16* o,
                   int B, int n_heads, int T, int w, int chunk_tiles, float* part, int* err, cudaStream_t st) {
  switch (dk) {
    case 16: return launch_attention_bf16<16>(qkv, mask, ek, ev, o, B, n_heads, T, w, chunk_tiles, part, err, st);
    case 32: return launch_attention_bf16<32>(qkv, mask, ek, ev, o, B, n_heads, T, w, chunk_tiles, part, err, st);
    case 48: return launch_attention_bf16<48>(qkv, mask, ek, ev, o, B, n_heads, T, w, chunk_tiles, part, err, st);
    case 64: return launch_attention_bf16<64>(qkv, mask, ek, ev, o, B, n_heads, T, w, chunk_tiles, part, err, st);
    case 96: return launch_attention_bf16<96>(qkv, mask, ek, ev, o, B, n_heads, T, w, chunk_tiles, part, err, st);
    case 128:   // refused by the shared-memory check on a B200
      return launch_attention_bf16<128>(qkv, mask, ek, ev, o, B, n_heads, T, w, chunk_tiles, part, err, st);
    default: return fail(VSG_EUNSUPPORTED, "attention head width %d (supported: 16, 32, 48, 64, 96)", dk);
  }
}
}  // namespace

// RelativeEncoder.forward (modules/rel_transformer.py:286-320) in the throughput mode: channels-last bf16 activations, the
// projections and the FFN on the tcgen05 convolution kernel (residual adds, ReLU and masks in its epilogue), attention on
// the tcgen05 kernel of attn_tc.cuh (split into key chunks of 2048 plus a combine beyond T = 2048), LayerNorm + condition
// + mask fused in one pass.
static int relenc_core_tc(const VsgPack* P, const float* x, const float* mask, const float* g, int g_t, int B, int T,
                          Workspace& ws, cudaStream_t st, __nv_bfloat16** xb_out, int** err_out) {
  const RelEncPack& e = P->relenc;
  const int H = e.hidden, F = e.filter, NL = e.n_layers, K = e.kernel, dk = H / e.n_heads;
  if (e.layers.empty() || !e.layers[0].qkv_tc.has_tmap || !e.layers[0].ffn1_tc.has_tmap || !e.layers[0].ffn2_tc.has_tmap ||
      H > 256 || (H & 1))
    return fail(VSG_EUNSUPPORTED, "bf16 encoder needs hidden / filter channels that are multiples of 16 (hidden <= 256)");
  typedef __nv_bfloat16 bf;
  bf* xb = ws.take<bf>((size_t)B * T * H);
  bf* ob = ws.take<bf>((size_t)B * T * H);
  bf* qkv = ws.take<bf>((size_t)B * T * 3 * H);
  bf* fb = ws.take<bf>((size_t)B * T * F);
  float* gp = ws.take<float>((size_t)B * H * (g_t ? T : 1));
  const int chunk_tiles = T > 128 * tc::kAtMaxTiles ? tc::kAtMaxTiles : 0;
  float* part = chunk_tiles ? ws.take<float>(attention_split_floats(B, T, e.n_heads, dk, chunk_tiles)) : nullptr;
  int* err = ws.take<int>(1);
  if (ws.overflow) return fail(VSG_ENOMEM, "encoder workspace too small: need %zu bytes", ws.off);
  VSG_CUDA_TRY(cudaMemsetAsync(err, 0, sizeof(int), st));
  if (g && e.gin <= 0) return fail(VSG_EINVAL, "this encoder has no pre_net (gin_channels is None) but g was given");
  const TCOptions opt = g_default_opts;
  const float* gadd = nullptr;
  if (g) {
    if (g_t) VSG_TRY(conv_f32_plain(e.pre_net, g, B, T, gp, st));
    else VSG_TRY(launch_cond(e.pre_w, e.pre_b, g, gp, H, e.gin, B, st));
    gadd = gp;
  }
  {
    dim3 grid((T + 31) / 32, (H + 31) / 32, B), block(32, 8);
    relenc_entry_bf16_kernel<<<grid, block, 0, st>>>(x, gadd, g_t, mask, xb, H, T);
    VSG_LAUNCH_CHECK("relenc_entry_bf16_kernel");
  }
  const long long rows = (long long)B * T;
  const unsigned ln_blocks = (unsigned)((rows + 7) / 8);
  for (int i = 0; i < NL; ++i) {
    const RelEncLayer& L = e.layers[i];
    {
      EpiTC ep;
      ep.bias = L.qkv_tc.bias; ep.out_raw = qkv;
      VSG_TRY(launch_conv_tc(P, L.qkv_tc, xb, B, T, 0, 1, T, 1, 0, T, ep, opt, err, st));
    }
    VSG_TRY(attention_bf16(dk, qkv, mask, L.ek, L.ev, ob, B, e.n_heads, T, e.window, chunk_tiles, part, err, st));
    {  // x = x + conv_o(attn)
      EpiTC ep;
      ep.bias = L.o_tc.bias; ep.add0 = xb; ep.out_raw = xb;
      VSG_TRY(launch_conv_tc(P, L.o_tc, ob, B, T, 0, 1, T, 1, 0, T, ep, opt, err, st));
    }
    relenc_layernorm_bf16_kernel<256><<<ln_blocks, 256, 0, st>>>(xb, L.g1, L.b1, nullptr, 0, mask, 1e-4f, H, T, rows);
    VSG_LAUNCH_CHECK("relenc_layernorm_bf16_kernel");
    {  // relu(conv_1(x * mask)) * mask
      EpiTC ep;
      ep.bias = L.ffn1_tc.bias; ep.mask = mask; ep.slope = 0.f; ep.out_act = fb;
      VSG_TRY(launch_conv_tc(P, L.ffn1_tc, xb, B, T, -(K / 2), 1, T, 1, 0, T, ep, opt, err, st));
    }
    {  // x = x + conv_2(.)
      EpiTC ep;
      ep.bias = L.ffn2_tc.bias; ep.add0 = xb; ep.out_raw = xb;
      VSG_TRY(launch_conv_tc(P, L.ffn2_tc, fb, B, T, 0, 1, T, 1, 0, T, ep, opt, err, st));
    }
    relenc_layernorm_bf16_kernel<256><<<ln_blocks, 256, 0, st>>>(xb, L.g2, L.b2, (i + 1 < NL) ? gadd : nullptr, g_t, mask, 1e-4f,
                                                                 H, T, rows);
    VSG_LAUNCH_CHECK("relenc_layernorm_bf16_kernel");
  }
  *xb_out = xb;
  *err_out = err;
  return VSG_OK;
}

int relenc_forward_tc(const VsgPack* P, const float* x, const float* mask, const float* g, int g_t, float* y, int B, int T,
                      Workspace& ws, cudaStream_t st) {
  __nv_bfloat16* xb = nullptr;
  int* err = nullptr;
  VSG_TRY(relenc_core_tc(P, x, mask, g, g_t, B, T, ws, st, &xb, &err));
  const int H = P->relenc.hidden;
  dim3 grid((T + 31) / 32, (H + 31) / 32, B), block(32, 8);
  transpose_from_bf16_kernel<<<grid, block, 0, st>>>(xb, y, H, T, 0, 1);
  VSG_LAUNCH_CHECK("transpose_from_bf16_kernel");
  return VSG_OK;
}

size_t frame_prior_ws_bytes(const VsgPack* P, int B, int T, int precision) {
  const RelEncPack& e = P->relenc;
  if (precision == VSG_PRECISION_BF16)
    return relenc_ws_bytes_tc(P, B, T, 1) + align256((size_t)B * T * 2 * e.hidden * 2) + align256((size_t)B * 2 * e.hidden * T * 4);
  return relenc_ws_bytes_f32(P, B, T, 1) + align256((size_t)B * e.hidden * T * sizeof(float));
}

// FramePriorNetwork.forward + prior sampling in the throughput mode: the encoder's channels-last bf16 output feeds proj
// (tcgen05, mask in the epilogue) without leaving that layout; stats -> fp32 [B, 2H, T]; z_p = (mu + noise exp(logs)) mask.
int frame_prior_forward_tc(const VsgPack* P, const float* x, const float* mask, const float* g, const float* noise,
                           float* stats, float* z, int B, int T, Workspace& ws, cudaStream_t st) {
  const RelEncPack& e = P->relenc;
  const int H = e.hidden;
  if (!e.proj_tc.has_tmap) return fail(VSG_EUNSUPPORTED, "bf16 frame prior needs hidden channels that are a multiple of 16");
  __nv_bfloat16* xb = nullptr;
  int* err = nullptr;
  VSG_TRY(relenc_core_tc(P, x, mask, g, g ? 1 : 0, B, T, ws, st, &xb, &err));
  __nv_bfloat16* sb = ws.take<__nv_bfloat16>((size_t)B * T * 2 * H);
  float* st32 = stats ? stats : ws.take<float>((size_t)B * 2 * H * T);
  if (ws.overflow) return fail(VSG_ENOMEM, "frame prior workspace too small: need %zu bytes", ws.off);
  {
    EpiTC ep;
    ep.bias = e.proj_tc.bias; ep.mask = mask; ep.out_raw = sb;
    VSG_TRY(launch_conv_tc(P, e.proj_tc, xb, B, T, 0, 1, T, 1, 0, T, ep, g_default_opts, err, st));
  }
  {
    dim3 grid((T + 31) / 32, (2 * H + 31) / 32, B), block(32, 8);
    transpose_from_bf16_kernel<<<grid, block, 0, st>>>(sb, st32, 2 * H, T, 0, 1);
    VSG_LAUNCH_CHECK("transpose_from_bf16_kernel");
  }
  const long long n = (long long)B * H * T;
  posterior_sample_from_stats_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(st32, noise, mask, z, H, T, n);
  VSG_LAUNCH_CHECK("posterior_sample_from_stats_kernel");
  return VSG_OK;
}

// ConvTranspose1d of decoder stage `us` (decoder.py:46) + its bias over nb utterances: out_act = leaky_relu(y) and, if
// given, out_raw = y and out_f32 = y, [nb, Lin * rate, Cout] channels-last.  merged: ONE Conv1d(Cin -> rate * Cout) over the
// input rate, whose [nb, Lin, rate * Cout] output is, byte for byte, the upsampled tensor; else one strided launch per
// polyphase.  x3: two bf16 planes per tensor.  out_part > 0: the output planes are planar, out_part elements apart (rows of
// Cout channels); 0: rows [hi | lo] (the merged form needs planar planes in x3).  in_ld / in_part: the input's layout as
// launch_conv_tc takes it (0 = rows [hi | lo]).
int launch_upsample_tc(const VsgPack* P, const UpStage& us, bool x3, bool merged, const __nv_bfloat16* xin, int nb, int Lin,
                       __nv_bfloat16* out_act, __nv_bfloat16* out_raw, float* out_f32, int out_part, int in_ld, int in_part,
                       const TCOptions& opt, int* err, cudaStream_t st, int* image_out = nullptr) {
  const int Lout = Lin * us.rate, ch = us.Cout;
  if (merged) {
    EpiTC e;
    e.bias = us.merged_tc.bias;
    e.out_act = out_act; e.out_raw = out_raw; e.out_f32 = out_f32;
    if (out_part) { e.ld = us.rate * ch; e.part_stride = out_part; }
    return launch_conv_tc(P, x3 ? us.merged_x3 : us.merged_tc, xin, nb, Lin, us.merged_in_off0, 1, Lin, 1, 0, Lin, e, opt, err,
                          st, in_ld, in_part, image_out);
  }
  for (int r = 0; r < us.rate; ++r) {   // one strided launch per polyphase
    EpiTC e;
    e.bias = us.phases[r].tc.bias;
    e.out_act = out_act; e.out_raw = out_raw; e.out_f32 = out_f32;
    if (out_part) { e.ld = ch; e.part_stride = out_part; }
    const int Lq = (Lout - r + us.rate - 1) / us.rate;
    VSG_TRY(launch_conv_tc(P, x3 ? us.phases[r].x3 : us.phases[r].tc, xin, nb, Lin, us.phases[r].in_off0, 1, Lq, us.rate, r,
                           Lout, e, opt, err, st, in_ld, in_part, image_out));
  }
  return VSG_OK;
}

// ---- L2-resident batch tiling --------------------------------------------------------------------------------
// Un-fused, one stage of the decoder streams 54 tensor passes through memory (SURVEY.md 7.2-3).  The stage tensors of
// ONE utterance are small (<= 9.6 MB in bf16), so each upsampling stage is run over sub-batches whose intermediates
// (x, leaky_relu(x), conv1 output, running resblock sum) stay in the 126 MB L2 between producer and consumer conv;
// they are overwritten by the next conv pair before they are ever evicted, so they never reach HBM.
struct SubBatchPlan { int sub[VSG_MAX_UPS]; size_t inter_elems; size_t io_elems; };

int g_l2_tensor_mb = 0;       // target size of one intermediate tensor of a sub-batch; 0 = off.  Measured on B200
                              // (round 1): with one kernel per conv the extra launches cost more than the L2 hits save
                              // (11.4 ms -> 16.0 ms per B16xT1000 step at 13 MB), so it is off until the fused kernels land.
int g_min_tiles = 592;        // keep >= 4 waves of 148 CTAs per launch when sub-batching

// T_plan > 0: the split of a T_plan-frame batch (a streaming window runs with the whole batch's split), buffers for T frames
SubBatchPlan plan_sub_batches(const VsgPack* P, int B, int T, int T_plan = 0) {
  SubBatchPlan pl;
  pl.inter_elems = 0;
  pl.io_elems = (size_t)B * P->cfg.dec_upsample_initial_channel * T;
  long long L = T, Lp = T_plan > 0 ? T_plan : T;
  for (size_t i = 0; i < P->ups.size(); ++i) {
    const UpStage& us = P->ups[i];
    L *= us.rate;
    Lp *= us.rate;
    const size_t per_utt = (size_t)us.Cout * (size_t)L;            // elements of one stage tensor of one utterance
    const size_t per_utt_p = (size_t)us.Cout * (size_t)Lp;
    const long long tiles_per_utt = (Lp + 127) / 128;
    long long sub = std::max<long long>(1, ((long long)g_l2_tensor_mb << 20) / (long long)(per_utt_p * 2));
    if (sub * tiles_per_utt < g_min_tiles) sub = (g_min_tiles + tiles_per_utt - 1) / tiles_per_utt;
    if (g_l2_tensor_mb <= 0 || sub * 2 > B) sub = B;               // not worth splitting
    static const int only_c = getenv("VSG_L2_ONLY_C") ? atoi(getenv("VSG_L2_ONLY_C")) : 0;   // A/B aid: sub-batch one stage width only
    if (only_c > 0 && us.Cout != only_c) sub = B;
    pl.sub[i] = (int)std::min<long long>(sub, B);
    pl.inter_elems = std::max(pl.inter_elems, per_utt * (size_t)pl.sub[i]);
    pl.io_elems = std::max(pl.io_elems, per_utt * (size_t)B);
  }
  return pl;
}

// The NK resblocks of a stage read the same input and only meet in the running sum, so their conv chains run on
// separate streams (chain 0 on the caller's stream): a persistent kernel's tail -- SMs idle while the last tiles finish,
// up to 14 % of the launch at C = 256 -- is filled by CTAs of the other chains.  Under CUDA-graph capture the fork / join
// events turn into graph edges.
// Helper streams and events belong to ONE (device, caller stream): two calls on different caller streams (two serving
// pipelines, two host threads) never share an event or a side stream, so the header's promise that a pack may be used
// from several streams of its device holds.  Calls on the SAME caller stream are ordered by that stream, as for any
// CUDA library.  The table is mutex-protected and bounded; beyond kMaxChainCtx distinct caller streams a call simply
// runs its chains back to back on its own stream.
constexpr int kMaxChains = 3;
constexpr size_t kMaxChainCtx = 256;
constexpr int kChainPool = 8;
struct ChainStreams {
  cudaStream_t s[kMaxChains - 1] = {nullptr, nullptr};
  cudaEvent_t fork = nullptr, join[kMaxChains - 1] = {nullptr, nullptr}, sum_done[kMaxChains] = {nullptr, nullptr, nullptr};
};
static std::mutex g_chain_mu;
static std::map<std::pair<int, cudaStream_t>, ChainStreams*> g_chain_ctx;   // bound contexts
static std::map<int, std::vector<ChainStreams*>> g_chain_free;               // created, not yet bound (per device)

static ChainStreams* chain_ctx_create() {
  ChainStreams* cs = new ChainStreams();
  bool ok = true;
  for (int i = 0; i < kMaxChains - 1 && ok; ++i)
    ok = cudaStreamCreateWithFlags(&cs->s[i], cudaStreamNonBlocking) == cudaSuccess &&
         cudaEventCreateWithFlags(&cs->join[i], cudaEventDisableTiming) == cudaSuccess;
  ok = ok && cudaEventCreateWithFlags(&cs->fork, cudaEventDisableTiming) == cudaSuccess;
  for (int i = 0; i < kMaxChains && ok; ++i) ok = cudaEventCreateWithFlags(&cs->sum_done[i], cudaEventDisableTiming) == cudaSuccess;
  if (ok) return cs;
  for (int i = 0; i < kMaxChains - 1; ++i) { if (cs->s[i]) cudaStreamDestroy(cs->s[i]); if (cs->join[i]) cudaEventDestroy(cs->join[i]); }
  if (cs->fork) cudaEventDestroy(cs->fork);
  for (int i = 0; i < kMaxChains; ++i) if (cs->sum_done[i]) cudaEventDestroy(cs->sum_done[i]);
  delete cs;
  cudaGetLastError();
  return nullptr;
}

// nullptr in *out (with VSG_OK) = no context available: the caller runs its chains back to back on its own stream.
// Streams and events are only ever CREATED outside graph capture (the first eager call on a device fills a small pool);
// a capturing stream binds a pooled context, so the warm-up-then-capture pattern of HotPathGraph keeps its chains.
static int chain_streams_for(int device, cudaStream_t caller, ChainStreams** out) {
  std::lock_guard<std::mutex> lock(g_chain_mu);
  *out = nullptr;
  const auto key = std::make_pair(device, caller);
  auto it = g_chain_ctx.find(key);
  if (it != g_chain_ctx.end()) { *out = it->second; return VSG_OK; }
  if (g_chain_ctx.size() >= kMaxChainCtx) return VSG_OK;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(caller, &cap) != cudaSuccess) { cudaGetLastError(); return VSG_OK; }
  std::vector<ChainStreams*>& pool = g_chain_free[device];
  if (cap == cudaStreamCaptureStatusNone)
    while ((int)pool.size() < kChainPool) {
      ChainStreams* cs = chain_ctx_create();
      if (!cs) break;
      pool.push_back(cs);
    }
  if (pool.empty()) return VSG_OK;
  ChainStreams* cs = pool.back();
  pool.pop_back();
  g_chain_ctx[key] = cs;
  *out = cs;
  return VSG_OK;
}

size_t dec_ws_bytes_tc(const VsgPack* P, int B, int T, bool x3, int T_plan) {
  const SubBatchPlan pl = plan_sub_batches(P, B, T, T_plan);
  const size_t np = x3 ? 2 : 1;
  return align256((size_t)B * T * P->cfg.dec_initial_channel * 2 * np) + align256((size_t)B * P->cfg.dec_upsample_initial_channel * 4) +
         2 * align256(pl.io_elems * 2 * np) + (7 + 4 * (kMaxChains - 1)) * align256(pl.inter_elems * 2 * np) + 512;
}

// ---- kernel choices of the decoder ---------------------------------------------------------------------------------
// Several choices depend on a stage's length, and the kernels they pick do not round alike: the row-packed and whole-
// resblock kernels keep the resblock residual in fp32 (TMEM), the per-convolution path stores it in bf16 between the
// convolutions; the fused pair rounds its intermediate like the per-convolution path but is only taken on long stages.  So
// every such choice is made from the WHOLE padded batch's stage length L (and its sub-batch nb): a streaming window
// (DecWin) runs the kernels the one-pass call runs, and if one of them cannot take the window's length the window is
// widened (dec_window_needs_tc) -- the kernel is never switched.
struct StageChoice { bool rb, rp, stage_planar; };

bool dec_one_stream(const TCOptions& opt, bool x3) {
  // Only leaky_relu(x) is stored for the running stream; split-bf16 recovers the residual from the two planes in fp32
  // (x = a >= 0 ? a : a / slope: as exact as a raw copy at ~16 mantissa bits) unless VSG_X3_TWO_STREAMS=1
  static const bool x3_two_streams = getenv("VSG_X3_TWO_STREAMS") != nullptr && getenv("VSG_X3_TWO_STREAMS")[0] == '1';
  return opt.single_stream && !(x3 && x3_two_streams);
}

StageChoice stage_choice(const VsgPack* P, int i, int B, int nb, int L, bool x3, const TCOptions& opt) {
  const VsgConfig& c = P->cfg;
  const UpStage& us = P->ups[i];
  const int ch = us.Cout, NK = c.dec_n_kernels;
  const bool one_stream_all = dec_one_stream(opt, x3);
  StageChoice sc;
  // C <= 64 stages: every ResBlock1 is ONE kernel (rb_tc.cuh); the three launches of a stage are chained through the
  // running sum, so they stay on the caller's stream (their CTAs own all of tensor memory and cannot co-reside anyway)
  sc.rb = c.dec_resblock == 1 && !x3 && opt.fuse_rb && ch <= 64;
  for (int j = 0; j < NK && sc.rb; ++j) {
    RbPlan rp;
    sc.rb = rb_plan(us.blocks[j], ch, L, opt, &rp) && L >= 256;
  }
  static const int rp_max_c_env = getenv("VSG_RP_MAX_C") ? atoi(getenv("VSG_RP_MAX_C")) : -1;   // A/B aid
  const int rp_max_c = rp_max_c_env >= 0 ? rp_max_c_env : opt.rp_max_c;
  // (bf16x3: the kernel's split-bf16 instantiation; it reads the single activated stream)
  // (its planar planes are addressed through the conv kernel's int part_stride: nb * L * ch must fit)
  sc.rp = c.dec_resblock == 1 && (x3 ? (opt.rp_x3 && one_stream_all && (size_t)nb * L * ch < ((size_t)1 << 31)) : true) &&
          opt.fuse_rp && ch <= rp_max_c;
  for (int j = 0; j < NK && sc.rp; ++j) {
    RpPlan rp;
    sc.rp = rp_plan(us.blocks[j], ch, L, opt, &rp, x3) && L >= 256;
  }
  // bf16x3 per-convolution ResBlock1 stages: every tensor of the stage planar through the conv kernel's ld / part_stride
  // (the stage output too, unless conv_post reads it): that is what lets them take the merged-polyphase upsampler as
  // well.  VSG_X3_PLANAR=0 (A/B aid): rows [hi | lo] as before
  static const bool x3_planar_on = !(getenv("VSG_X3_PLANAR") && getenv("VSG_X3_PLANAR")[0] == '0');
  sc.stage_planar = x3 && !sc.rp && x3_planar_on && one_stream_all && c.dec_resblock == 1 && !sc.rb && nb == B &&
                    i + 1 < c.dec_n_ups && (size_t)nb * L * ch < ((size_t)1 << 31);
  return sc;
}

// measured on B200 (tools/time_pair.py, B=16): C=32 pair 156-204 us vs 188-241 us un-fused; at C=16 the single epilogue
// warp set of the one-CTA-per-SM pair kernel is slower (239-275 us) than two co-resident un-fused CTAs (210-235 us), so
// only C=32 is fused by default (fuse_pairs == 2 forces both).
bool pair_choice(const VsgPack* P, const ResBlockPack& rb, int q, int ch, int L, bool x3, const TCOptions& opt, bool has_add1,
                 int n_outs) {
  return P->cfg.dec_resblock == 1 && !x3 && opt.fuse_pairs && (ch == 32 || ch == 16 || opt.fuse_pairs == 2) &&
         pair_supported(rb.c1_tc[q], rb.c2_tc[q], rb.dilations[q], L, 1 + (has_add1 ? 1 : 0), n_outs);
}

// conv_post: 0 tcgen05, rows of 4 samples | 1 register-window kernel | 2 shared-memory-window kernel (A/B aids) |
// 3 tcgen05 bf16x3, rows of 2 samples | 4 one thread per sample
int post_choice(const VsgPack* P, int ch, int L, bool x3, const TCOptions& opt) {
  if (!x3 && ch == 16 && P->conv_post_k == 7) {   // the model's shape
    if (opt.conv_post == 0 && P->conv_post_S == 4 && L % 4 == 0) return 0;
    return opt.conv_post == 1 ? 1 : 2;
  }
  if (x3 && ch == 16 && P->conv_post_k == 7 && P->conv_post_rp_x3.has_tmap && L % 2 == 0 && opt.conv_post == 0) return 3;
  return 4;
}

int dec_window_needs_tc(const VsgPack* P, int B, int T, bool x3, int* min_frames, int* align) {
  const VsgConfig& c = P->cfg;
  const TCOptions opt = g_default_opts;
  const SubBatchPlan pl = plan_sub_batches(P, B, T);
  const bool one_stream = dec_one_stream(opt, x3);
  int need = 1, A = 1;
  long long R = 1;                               // samples per frame at the current stage
  auto min_len = [&](long long Lmin) { need = std::max(need, (int)((Lmin + R - 1) / R)); };
  // a kernel with S time steps per row sums each output in an order set by its row phase: windows start and end where
  // the one-pass call has phase 0, i.e. on multiples of S / gcd(S, R) frames
  auto row_phase = [&](int S) { const int a = S / (int)std::gcd((long long)S, R); A = A / std::gcd(A, a) * a; };
  int ch = c.dec_upsample_initial_channel;
  for (int i = 0; i < c.dec_n_ups; ++i) {
    const UpStage& us = P->ups[i];
    R *= us.rate;
    ch = us.Cout;
    const int L = (int)(T * R);
    for (int b0 = 0; b0 < B; b0 += pl.sub[i]) {
      const int nb = std::min(pl.sub[i], B - b0);
      const StageChoice sc = stage_choice(P, i, B, nb, L, x3, opt);
      if (sc.rb) min_len(256);
      if (sc.rp) { min_len(256); row_phase(64 / ch); }
      if (sc.rb || sc.rp) continue;
      for (int j = 0; j < c.dec_n_kernels; ++j) {
        const ResBlockPack& rb = us.blocks[j];
        const int nd = (int)rb.dilations.size();
        for (int q = 0; q < nd; ++q) {
          const bool last = q == nd - 1;
          if (pair_choice(P, rb, q, ch, L, x3, opt, last && j > 0, last ? 1 : (one_stream ? 1 : 2))) min_len(128 * pair_mb(ch));
        }
      }
    }
  }
  const int post = post_choice(P, ch, (int)(T * R), x3, opt);
  if (post == 1) return fail(VSG_EUNSUPPORTED, "the register-window conv_post kernel (tuning option) has no window form");
  if (post == 0) row_phase(4);
  if (post == 3) row_phase(2);
  *min_frames = std::min(need, T);
  *align = A;
  return VSG_OK;
}

// Generator.forward (modules/visinger/decoder.py:40-59) on the tensor-core kernels.
// x3: split-bf16 mode -- every activation tensor carries two bf16 planes [hi | lo] per row and every product is
// three MMAs (hi*W_hi + hi*W_lo + lo*W_hi): fp32-tolerance results on the tensor cores.
int generator_forward_tc(const VsgPack* P, const float* z, const float* g, float* wav, int B, int T, Workspace& ws,
                         cudaStream_t st, bool x3, const DecWin* win) {
  const VsgConfig& c = P->cfg;
  const int C0 = c.dec_initial_channel, UIC = c.dec_upsample_initial_channel, NK = c.dec_n_kernels;
  if (!P->conv_pre_tc.has_tmap) return fail(VSG_EUNSUPPORTED, "bf16 decoder needs channel counts that are multiples of 16");
  const int T_plan = win ? win->T_plan : T;     // every length-dependent kernel choice below is made from the whole batch
  const SubBatchPlan pl = plan_sub_batches(P, B, T, T_plan);
  typedef __nv_bfloat16 bf;
  const size_t np = x3 ? 2 : 1;             // bf16 planes per activation tensor
  auto W = [&](const ConvWTC& plain, const ConvWTC& split) -> const ConvWTC& { return x3 ? split : plain; };
  bf* zt = ws.take<bf>((size_t)B * T * C0 * np);
  float* cond = ws.take<float>((size_t)B * UIC);
  bf* io[2] = {ws.take<bf>(pl.io_elems * np), ws.take<bf>(pl.io_elems * np)};   // leaky_relu'd stage input / output
  bf* bU = ws.take<bf>(pl.inter_elems * np);    // upsampled x (residual for the first pair of every resblock)
  bf* bUA = ws.take<bf>(pl.inter_elems * np);   // leaky_relu(x)
  // per resblock chain (they run concurrently): running x, leaky_relu of it, leaky_relu(conv1 output), its ResBlock2 partner
  bf *cR[kMaxChains], *cRA[kMaxChains], *cT[kMaxChains], *cTA[kMaxChains];
  for (int j = 0; j < kMaxChains; ++j) {
    cR[j] = ws.take<bf>(pl.inter_elems * np);
    cRA[j] = ws.take<bf>(pl.inter_elems * np);
    cT[j] = ws.take<bf>(pl.inter_elems * np);
    cTA[j] = ws.take<bf>(pl.inter_elems * np);
  }
  bf* bS = ws.take<bf>(pl.inter_elems * np);    // running sum over the NK resblocks
  int* err = ws.take<int>(1);
  if (ws.overflow) return fail(VSG_ENOMEM, "generator workspace too small: need %zu bytes", ws.off);
  VSG_CUDA_TRY(cudaMemsetAsync(err, 0, sizeof(int), st));
  const TCOptions opt = g_default_opts;
  bool chains = opt.chain_streams && NK > 1 && NK <= kMaxChains;
  ChainStreams* cs = nullptr;
  if (chains) {
    VSG_TRY(chain_streams_for(P->device, st, &cs));
    if (!cs) chains = false;
  }

  if (c.dec_gin > 0) {
    if (!g) return fail(VSG_EINVAL, "generator was built with gin_channels=%d but g is NULL", c.dec_gin);
    VSG_TRY(launch_cond(P->dec_cond_w, P->dec_cond_b, g, cond, UIC, c.dec_gin, B, st));
  }
  {  // boundary: [B, C, T] fp32 -> [B, T, C] bf16, once
    dim3 grid((T + 31) / 32, (C0 + 31) / 32, B), block(32, 8);
    transpose_to_bf16_kernel<<<grid, block, 0, st>>>(z, zt, C0, T, x3 ? 2 : 1, nullptr, nullptr, nullptr, win ? win->z_ld : 0);
    VSG_LAUNCH_CHECK("transpose_to_bf16_kernel");
  }
  int cur_io = 0;
  {  // x = conv_pre(z) + cond(g); only leaky_relu(x) is ever consumed (decoder.py:41-45)
    EpiTC e;
    e.bias = P->conv_pre_tc.bias;
    if (c.dec_gin > 0) { e.bcond = cond; e.bcond_bs = UIC; }
    e.out_act = io[cur_io];
    VSG_TRY(launch_conv_tc(P, W(P->conv_pre_tc, P->conv_pre_x3), zt, B, T, -3, 1, T, 1, 0, T, e, opt, err, st));
  }
  // Only leaky_relu(x) is stored for the running stream (see below and dec_one_stream)
  const bool one_stream_all = dec_one_stream(opt, x3);
  int L = T, ch = UIC;
  long long Lp = T_plan;                      // the stage length of the whole batch: the kernel choices' length
  bool prev_planar = false;                   // bf16x3: the stage input is a planar two-plane tensor
  for (int i = 0; i < c.dec_n_ups; ++i) {
    const UpStage& us = P->ups[i];
    const int Lin = L, Cin = ch, Lout = L * us.rate;
    ch = us.Cout; L = Lout;
    Lp *= us.rate;
    const bf* stage_in = io[cur_io];
    bf* stage_out = io[cur_io ^ 1];
    bool stage_planar_out = false;
    for (int b0 = 0; b0 < B; b0 += pl.sub[i]) {
      const int nb = std::min(pl.sub[i], B - b0);
      const bf* xin = stage_in + (size_t)b0 * Lin * Cin * (prev_planar ? 1 : np);   // (planar: plane 0 of utterance b0)
      bf* xout = stage_out + (size_t)b0 * L * ch * np;
      const StageChoice sc = stage_choice(P, i, B, nb, (int)Lp, x3, opt);
      const bool rb_stage = sc.rb, rp_stage = sc.rp;
      // bf16x3 row-packed stages: the upsampler writes its two planes PLANAR ([2][nb, L, ch]: each plane is then an
      // ordinary one-plane tensor for the resblock kernel's row-packed tensor map), as is the running resblock sum;
      // the per-convolution ResBlock1 stages of the bf16x3 mode are planar too (stage_choice)
      const bool planar = x3 && rp_stage;
      const bool stage_planar = sc.stage_planar;
      const bool planar_any = planar || stage_planar;
      stage_planar_out = stage_planar;
      const int up_ld = planar_any ? ch : 0, up_part = planar_any ? (int)((size_t)nb * L * ch) : 0;
      // the stage input is planar if the previous stage wrote it so: that stage ran whole (nb == B), so its planes are
      // B * Lin * Cin elements apart whatever this stage's sub-batches are
      const int in_ld = prev_planar ? Cin : 0, in_part = prev_planar ? (int)((size_t)B * Lin * Cin) : 0;
      // (split-bf16 planes interleaved per row would come out wrong; PLANAR planes are one-plane tensors each, so the
      // bf16x3 row-packed stages take the merged form too)
      static const bool x3_merge_off = getenv("VSG_X3_NO_MERGED_UPS") != nullptr;   // A/B aid
      const bool merged = opt.merge_ups && (!x3 || (planar_any && us.merged_x3.has_tmap && !x3_merge_off)) &&
                          us.merged_tc.has_tmap && Lout == Lin * us.rate;
      VSG_TRY(launch_upsample_tc(P, us, x3, merged, xin, nb, Lin, bUA, one_stream_all ? nullptr : bU, nullptr, up_part, in_ld,
                                 in_part, opt, err, st));
      // Only leaky_relu(x) is stored for the running stream; the residual x is recovered from it in the consumer's
      // epilogue (a > 0 ? a : a / slope -- as exact as a second, raw copy at the stream's precision), so the upsampler and
      // every non-final conv2 write one tensor instead of two.
      const bool one_stream = one_stream_all;
      const cudaStream_t st_main = st;
      if (rb_stage || rp_stage) {
        for (int j = 0; j < NK; ++j) {        // xs = sum_j resblock_j(x); x = xs / NK (decoder.py:47-54)
          const bool lastj = (j == NK - 1);
          if (rp_stage)
            VSG_TRY(launch_rp_tc(P, us.blocks[j], ch, bUA, nb, L, j > 0 ? bS : nullptr, lastj ? nullptr : bS, lastj ? xout : nullptr,
                                 nullptr, lastj ? 1.0f / (float)NK : 1.0f, opt, err, st, x3));
          else
            VSG_TRY(launch_rb_tc(P, us.blocks[j], ch, bUA, nb, L, j > 0 ? bS : nullptr, lastj ? nullptr : bS, lastj ? xout : nullptr,
                                 nullptr, lastj ? 1.0f / (float)NK : 1.0f, opt, err, st));
        }
        continue;
      }
      // A/B aid: VSG_CHAIN_MIN_C = narrowest stage whose resblock chains run on separate streams (read per call)
      const char* cmc = getenv("VSG_CHAIN_MIN_C");
      const bool chains_st = chains && (!cmc || ch >= atoi(cmc));
      if (chains_st) {   // fork: the other chains start once the upsampled input is complete
        VSG_CUDA_TRY(cudaEventRecord(cs->fork, st_main));
        for (int j = 1; j < NK; ++j) VSG_CUDA_TRY(cudaStreamWaitEvent(cs->s[j - 1], cs->fork, 0));
      }
      // every failure between fork and join must still join the side streams (a capture would otherwise be left with
      // un-joined branches), so the chains run inside a lambda and the join below is unconditional
      auto run_resblocks = [&]() -> int {
      for (int j = 0; j < NK; ++j) {        // xs = sum_j resblock_j(x); x = xs / NK (decoder.py:47-54)
        const ResBlockPack& rb = us.blocks[j];
        const int nd = (int)rb.dilations.size(), k = rb.kernel;
        const bf* cur = one_stream ? bUA : bU; const bf* curA = bUA;
        const int cj = chains_st ? j : 0;
        bf *bR = cR[cj], *bRA = cRA[cj], *bT = cT[cj], *bTA = cTA[cj];
        if (chains_st) st = j == 0 ? st_main : cs->s[j - 1];
        for (int q = 0; q < nd; ++q) {
          const bool last = (q == nd - 1);
          const int d = rb.dilations[q];
          // the running sum is read-modify-written by the last conv of every chain, in chain order
          const bool sum_wait = chains_st && last && j > 0;
          EpiTC e2;
          e2.add0 = cur;
          e2.add0_is_act = one_stream ? 1 : 0;
          if (last) {
            e2.add1 = (j > 0) ? bS : nullptr;
            if (j == NK - 1) { e2.scale = 1.0f / (float)NK; e2.out_act = xout; }
            else e2.out_raw = bS;
          }
          const int n_outs_pair = last ? 1 : (one_stream ? 1 : 2);
          const bool fuse = pair_choice(P, rb, q, ch, (int)Lp, x3, opt, e2.add1 != nullptr, n_outs_pair);
          if (fuse) {
            // low-channel stages: both convs of the pair in ONE kernel, the intermediate never leaves the SM
            // The pair kernel reads its input with a halo (rows of the NEIGHBOUR tiles) while other CTAs store their
            // output tiles: it must never run in place.  The running stream ping-pongs between the chain's R and T buffers
            // (the T buffers are otherwise unused on the fused path).
            e2.bias = rb.c2_tc[q].bias;
            bf* nr = (curA == bRA) ? bT : bR;
            bf* nra = (curA == bRA) ? bTA : bRA;
            if (!last) { e2.out_act = nra; if (!one_stream) e2.out_raw = nr; }
            if (sum_wait) VSG_CUDA_TRY(cudaStreamWaitEvent(st, cs->sum_done[j - 1], 0));
            VSG_TRY(launch_pair_tc(P, rb.c1_tc[q], rb.c2_tc[q], curA, nb, L, d, e2, opt, err, st));
            cur = one_stream ? nra : nr; curA = nra;
          } else if (c.dec_resblock == 1) {        // ResBlock1 (decoder.py:91-104)
            // conv1 writes a scratch tensor of the OTHER buffer pair; conv2 reads that scratch (with a halo) and updates
            // the running stream, in place when it already lives in this chain's buffers: its add0 / output tiles are
            // the same rows of the same CTA, so only the scratch is ever read across tile borders.
            const bool in_t = (curA == bTA);          // a preceding fused pair may have left the stream in the T pair
            bf* tmp = in_t ? bR : bT;
            bf* nr = in_t ? bT : bR;
            bf* nra = in_t ? bTA : bRA;
            EpiTC e1;
            e1.bias = rb.c1_tc[q].bias; e1.out_act = tmp;
            if (stage_planar) { e1.ld = ch; e1.part_stride = up_part; e2.ld = ch; e2.part_stride = up_part; }
            VSG_TRY(launch_conv_tc(P, W(rb.c1_tc[q], rb.c1_x3[q]), curA, nb, L, -((k * d - d) / 2), d, L, 1, 0, L, e1, opt, err, st,
                                   up_ld, up_part));
            e2.bias = rb.c2_tc[q].bias;
            if (!last) { e2.out_act = nra; if (!one_stream) e2.out_raw = nr; }
            if (sum_wait) VSG_CUDA_TRY(cudaStreamWaitEvent(st, cs->sum_done[j - 1], 0));
            VSG_TRY(launch_conv_tc(P, W(rb.c2_tc[q], rb.c2_x3[q]), tmp, nb, L, -((k - 1) / 2), 1, L, 1, 0, L, e2, opt, err, st,
                                   up_ld, up_part));
            cur = one_stream ? nra : nr; curA = nra;
          } else {                           // ResBlock2 (decoder.py:124-133)
            e2.bias = rb.c1_tc[q].bias;
            bf* nr = (cur == bR || cur == bRA) ? bT : bR;
            bf* nra = (cur == bR || cur == bRA) ? bTA : bRA;
            if (!last) { e2.out_act = nra; if (!one_stream) e2.out_raw = nr; }
            if (sum_wait) VSG_CUDA_TRY(cudaStreamWaitEvent(st, cs->sum_done[j - 1], 0));
            VSG_TRY(launch_conv_tc(P, W(rb.c1_tc[q], rb.c1_x3[q]), curA, nb, L, -((k * d - d) / 2), d, L, 1, 0, L, e2, opt, err, st));
            cur = one_stream ? nra : nr; curA = nra;
          }
        }
        if (chains_st && j < NK - 1) VSG_CUDA_TRY(cudaEventRecord(cs->sum_done[j], st));
      }
      return VSG_OK;
      };
      const int rc_chains = run_resblocks();
      if (chains_st) {   // join: the stage output (written by the last chain) and every scratch buffer are settled
        st = st_main;
        cudaError_t je = cudaSuccess;
        for (int j = 1; j < NK; ++j) {
          cudaError_t e1 = cudaEventRecord(cs->join[j - 1], cs->s[j - 1]);
          cudaError_t e2 = e1 == cudaSuccess ? cudaStreamWaitEvent(st_main, cs->join[j - 1], 0) : e1;
          if (je == cudaSuccess) je = e2;
        }
        if (rc_chains == VSG_OK && je != cudaSuccess)
          return fail(VSG_ECUDA, "joining the resblock chains failed: %s", cudaGetErrorString(je));
      }
      VSG_TRY(rc_chains);
    }
    cur_io ^= 1;
    prev_planar = stage_planar_out;
  }
  {  // wav = tanh(conv_post(leaky_relu(x)))   (decoder.py:55-57); the stage output already holds leaky_relu(x)
    // (a window: only its central samples [s0, s1) are computed or stored, straight into the caller's rows)
    const int post = post_choice(P, ch, (int)Lp, x3, opt);
    if (win && post == 1) return fail(VSG_EUNSUPPORTED, "the register-window conv_post kernel (tuning option) has no window form");
    if (post == 0 || post == 1 || post == 2) {   // the model's shape (16 channels, k = 7)
      constexpr int S = 8;
      if (post == 0) {
        // conv_post on the tensor cores: rows of 4 samples x 16 channels, Conv1d(64 -> 16, 3 row taps), tanh epilogue
        EpiTC e;
        e.mode = EPI_TC_TANH; e.out_f32 = wav; e.tanh_cols = 4;
        if (win) { e.tanh_ld = win->wav_ld; e.tanh_s0 = win->s0; e.tanh_s1 = win->s1; }
        VSG_TRY(launch_conv_tc(P, P->conv_post_rp, io[cur_io], B, L / 4, -1, 1, L / 4, 1, 0, L / 4, e, opt, err, st));
      } else if (post == 1) {
        const int gpb = (L + S - 1) / S, total = gpb * B;
        const int blocks = std::min((total + 127) / 128, 8 * P->sm_count);
        conv_post_bf16_win_kernel<16, 7, S><<<blocks, 128, 0, st>>>(io[cur_io], P->conv_post_w, wav, L, gpb, total);
        VSG_LAUNCH_CHECK("conv_post_bf16_win_kernel");
      } else {
        const int tpb = (L + 128 * S - 1) / (128 * S), total = tpb * B;
        const int blocks = std::min(total, 6 * P->sm_count);
        conv_post_bf16_smem_kernel<16, 7, S><<<blocks, 128, 0, st>>>(io[cur_io], P->conv_post_w, wav, L, tpb, total,
                                                                    win ? win->s0 : 0, win ? win->s1 : 0, win ? win->wav_ld : 0);
        VSG_LAUNCH_CHECK("conv_post_bf16_smem_kernel");
      }
    } else if (post == 3) {
      // bf16x3: rows of 2 samples x [hi | lo] x 16 channels, Conv1d(64 -> 16, 5 row taps) on [W_hi | W_lo], tanh epilogue
      EpiTC e;
      e.mode = EPI_TC_TANH; e.out_f32 = wav; e.tanh_cols = 2;
      if (win) { e.tanh_ld = win->wav_ld; e.tanh_s0 = win->s0; e.tanh_s1 = win->s1; }
      VSG_TRY(launch_conv_tc(P, P->conv_post_rp_x3, io[cur_io], B, L / 2, -2, 1, L / 2, 1, 0, L / 2, e, opt, err, st));
    } else {
      const int n0 = win ? win->s0 : 0, n1 = win ? win->s1 : L;
      dim3 grid((n1 - n0 + 255) / 256, B);
      conv_post_bf16_kernel<<<grid, 256, (size_t)ch * P->conv_post_k * sizeof(float), st>>>(
          io[cur_io], P->conv_post_w, wav, ch, L, P->conv_post_k, x3 ? 1 : 0, n0, n1, win ? win->wav_ld : 0);
      VSG_LAUNCH_CHECK("conv_post_bf16_kernel");
    }
  }
  return VSG_OK;
}

}  // namespace vsg

using namespace vsg;

// Per-layer parity hook (tests only; allocates and synchronises): one bf16 tensor-core Conv1d with the full
// fused epilogue.  See include/visinger_b200.h.
static TCOptions g_debug_force;      // plan override + repetitions for the next vsg_debug_conv1d_bf16 calls
static int g_debug_reps = 1;
static float g_debug_ms = 0.f;

extern "C" int vsg_debug_set_plan(int32_t mb, int32_t cw, int32_t two, int32_t resident, int32_t reps) {
  g_debug_force.force_mb = mb; g_debug_force.force_cw = cw; g_debug_force.force_two = two;
  g_debug_force.force_resident = resident;
  g_debug_reps = reps > 0 ? reps : 1;
  return VSG_OK;
}
extern "C" float vsg_debug_last_ms(void) { return g_debug_ms; }

extern "C" int vsg_debug_conv1d_bf16(const void* x_bf16, const float* w, const float* bias, const void* add0_bf16,
                                     const void* add1_bf16, float scale, float* out_f32, void* out_raw_bf16,
                                     void* out_act_bf16, int32_t B, int32_t L, int32_t Cin, int32_t Cout, int32_t k,
                                     int32_t dilation, int32_t flags, int32_t device) {
  reset_launch_counts();
  if (!x_bf16 || !w) return fail(VSG_EINVAL, "null pointer");
  VSG_CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  VSG_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  VsgPack tmp;
  tmp.device = device;
  tmp.sm_count = prop.multiProcessorCount;
  std::vector<float> W(w, w + (size_t)Cout * Cin * k), bz(Cout, 0.f);
  if (bias) bz.assign(bias, bias + Cout);
  ConvWTC wt;
  int rc = pack_conv_tc(&tmp, W, bz, Cout, Cin, k, &wt, (flags & 256) ? 3 : (flags & 4) ? 2 : 1);   // bit 8: three planes
  int* err = nullptr;
  if (rc == VSG_OK && cudaMalloc(&err, sizeof(int)) != cudaSuccess) rc = fail(VSG_ECUDA, "cudaMalloc failed");
  if (rc == VSG_OK) {
    cudaMemset(err, 0, sizeof(int));
    EpiTC e;
    e.bias = wt.bias;
    e.add0 = (const __nv_bfloat16*)add0_bf16;
    e.add1 = (const __nv_bfloat16*)add1_bf16;
    e.add0_is_act = (flags >> 3) & 1;
    e.scale = scale;
    e.out_f32 = out_f32;
    e.out_raw = (__nv_bfloat16*)out_raw_bf16;
    e.out_act = (__nv_bfloat16*)out_act_bf16;
    TCOptions opt;
    opt.halo_mode = flags & 1;
    opt.w_resident = (flags >> 1) & 1;
    opt.max_mb = ((flags >> 4) & 15) ? ((flags >> 4) & 15) : 4;
    opt.force_mb = g_debug_force.force_mb; opt.force_cw = g_debug_force.force_cw;
    opt.force_two = g_debug_force.force_two; opt.force_resident = g_debug_force.force_resident;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    rc = launch_conv_tc(&tmp, wt, (const __nv_bfloat16*)x_bf16, B, L, -((k - 1) * dilation / 2), dilation, L, 1, 0, L, e,
                        opt, err, 0);                                  // warm-up + correctness run
    if (rc == VSG_OK && g_debug_reps > 1) {
      cudaEventRecord(e0, 0);
      for (int r = 0; r < g_debug_reps && rc == VSG_OK; ++r)
        rc = launch_conv_tc(&tmp, wt, (const __nv_bfloat16*)x_bf16, B, L, -((k - 1) * dilation / 2), dilation, L, 1, 0, L,
                            e, opt, err, 0);
      cudaEventRecord(e1, 0);
    }
    if (rc == VSG_OK) {
      cudaError_t ce = cudaDeviceSynchronize();
      if (ce != cudaSuccess) rc = fail(VSG_ECUDA, "conv_tc_kernel execution failed: %s", cudaGetErrorString(ce));
      else if (g_debug_reps > 1) { cudaEventElapsedTime(&g_debug_ms, e0, e1); g_debug_ms /= g_debug_reps; }
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
  }
  if (err) cudaFree(err);
  for (void* q : tmp.allocs) cudaFree(q);
  return rc;
}

// One launch of conv_tc_kernel with every EpiTC field and every output geometry (tests only; allocates and synchronises).
// See include/visinger_b200.h.
extern "C" int vsg_debug_conv_tc(const VsgDebugConv* d, int32_t* image_out, int32_t device) {
  reset_launch_counts();
  if (!d || !d->x || !d->w) return fail(VSG_EINVAL, "vsg_debug_conv_tc: null descriptor, input or weight");
  if (d->planes < 1 || d->planes > 3) return fail(VSG_EINVAL, "vsg_debug_conv_tc: planes must be 1, 2 or 3");
  if (d->mode != EPI_TC_LINEAR && d->mode != EPI_TC_GATE && d->mode != EPI_TC_COUPLE)
    return fail(VSG_EINVAL, "vsg_debug_conv_tc: mode must be linear (0), gate (1) or couple (2)");
  if (d->epi_sigs < 0 || d->epi_sigs > 2) return fail(VSG_EINVAL, "vsg_debug_conv_tc: epi_sigs must be 0, 1 or 2");
  if (d->B <= 0 || d->Lin <= 0 || d->Cin <= 0 || d->Cout <= 0 || d->k <= 0 || d->dil <= 0 || d->Lq <= 0 || d->Lout <= 0 ||
      d->out_stride <= 0 || d->out_phase < 0 || d->out_phase >= d->out_stride || (d->Lq - 1) * d->out_stride + d->out_phase >= d->Lout)
    return fail(VSG_EINVAL, "vsg_debug_conv_tc: bad shape or output geometry");
  DebugScope sc;
  VSG_TRY(sc.open(device));
  std::vector<float> W(d->w, d->w + (size_t)d->Cout * d->Cin * d->k), bz(d->Cout, 0.f);
  if (d->bias) bz.assign(d->bias, d->bias + d->Cout);
  ConvWTC wt;
  VSG_TRY(pack_conv_tc(&sc.P, W, bz, d->Cout, d->Cin, d->k, &wt, d->planes));
  EpiTC e;
  e.mode = d->mode; e.mask = d->mask; e.couple_sign = d->couple_sign;
  e.ld = d->ld; e.part_stride = d->part_stride;
  e.add0_is_act = d->add0_is_act;
  e.bias = d->bias ? wt.bias : nullptr;
  e.bcond = d->bcond; e.bcond_bs = d->bcond_bs;
  e.add0 = (const __nv_bfloat16*)d->add0; e.add1 = (const __nv_bfloat16*)d->add1;
  e.scale = d->scale; e.slope = d->slope;
  e.out_raw = (__nv_bfloat16*)d->out_raw; e.out_act = (__nv_bfloat16*)d->out_act; e.out_f32 = d->out_f32;
  TCOptions opt;
  opt.epi_sigs = d->epi_sigs;
  int img = -1;
  const int rc = launch_conv_tc(&sc.P, wt, (const __nv_bfloat16*)d->x, d->B, d->Lin, d->in_off0, d->dil, d->Lq, d->out_stride,
                                d->out_phase, d->Lout, e, opt, sc.err, 0, d->x_ld, d->x_part_stride, &img);
  if (image_out) *image_out = img;
  return sc.finish(rc);
}

// The decoder's upsampler (ConvTranspose1d + bias + leaky_relu) as the generator launches it (tests only; allocates and
// synchronises).  See include/visinger_b200.h.
extern "C" int vsg_debug_upsample_tc(const void* x_bf16, const float* w, const float* bias, int32_t Cin, int32_t Cout,
                                     int32_t rate, int32_t k, int32_t B, int32_t Lin, void* out_act_bf16, void* out_raw_bf16,
                                     float* out_f32, int32_t flags, int32_t* image_out, int32_t device) {
  reset_launch_counts();
  if (!x_bf16 || !w || !bias || !out_act_bf16) return fail(VSG_EINVAL, "vsg_debug_upsample_tc: null input, weight, bias or output");
  if (Cin <= 0 || Cout <= 0 || B <= 0 || Lin <= 0) return fail(VSG_EINVAL, "vsg_debug_upsample_tc: bad shape");
  const bool merged = flags & 1, x3 = flags & 2, planar_in = flags & 4, planar_out = flags & 8;
  if (!x3 && (planar_in || planar_out)) return fail(VSG_EINVAL, "vsg_debug_upsample_tc: planar layouts need two planes");
  if (merged && x3 && !planar_out) return fail(VSG_EINVAL, "vsg_debug_upsample_tc: the two-plane merged form writes planar planes");
  const size_t in_part = (size_t)B * Lin * Cin, out_part = (size_t)B * Lin * rate * Cout;
  if (out_part >= ((size_t)1 << 31)) return fail(VSG_EINVAL, "vsg_debug_upsample_tc: tensor too large");
  DebugScope sc;
  VSG_TRY(sc.open(device));
  UpStage us;
  std::vector<float> W(w, w + (size_t)Cin * Cout * k), b(bias, bias + Cout);
  VSG_TRY(pack_upsampler(&sc.P, W, b, Cin, Cout, rate, k, &us));
  if (!(merged ? us.merged_tc.has_tmap : us.phases[0].tc.has_tmap))
    return fail(VSG_EUNSUPPORTED, "vsg_debug_upsample_tc: channel counts must be multiples of 16");
  TCOptions opt;
  int img = -1;
  const int rc = launch_upsample_tc(&sc.P, us, x3, merged, (const __nv_bfloat16*)x_bf16, B, Lin, (__nv_bfloat16*)out_act_bf16,
                                    (__nv_bfloat16*)out_raw_bf16, out_f32, planar_out ? (int)out_part : 0,
                                    planar_in ? Cin : 0, planar_in ? (int)in_part : 0, opt, sc.err, 0, &img);
  if (image_out) *image_out = img;
  return sc.finish(rc);
}

// Per-layer parity hook for the fused ResBlock1 pair (tests only; allocates and synchronises).
//   xa: device bf16 [B, L, C] = leaky_relu(x); w1/w2: HOST fp32 [C][C][k]; b1/b2: HOST fp32 [C]; add0/add1 as above;
//   v = (conv1d(leaky_relu(conv1d(xa, w1, dilation d1) + b1), w2) + b2 + add0 + add1) * scale.
extern "C" int vsg_debug_pair_bf16(const void* xa_bf16, const float* w1, const float* b1, const float* w2, const float* b2,
                                   const void* add0_bf16, const void* add1_bf16, float scale, float* out_f32,
                                   void* out_raw_bf16, void* out_act_bf16, int32_t B, int32_t L, int32_t C, int32_t k,
                                   int32_t d1, int32_t device) {
  reset_launch_counts();
  if (!xa_bf16 || !w1 || !w2 || !b1 || !b2) return fail(VSG_EINVAL, "null pointer");
  VSG_CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  VSG_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  VsgPack tmp;
  tmp.device = device;
  tmp.sm_count = prop.multiProcessorCount;
  std::vector<float> W1(w1, w1 + (size_t)C * C * k), W2(w2, w2 + (size_t)C * C * k), B1(b1, b1 + C), B2(b2, b2 + C);
  ConvWTC wt1, wt2;
  int rc = pack_conv_tc(&tmp, W1, B1, C, C, k, &wt1);
  if (rc == VSG_OK) rc = pack_conv_tc(&tmp, W2, B2, C, C, k, &wt2);
  int* err = nullptr;
  if (rc == VSG_OK && cudaMalloc(&err, sizeof(int)) != cudaSuccess) rc = fail(VSG_ECUDA, "cudaMalloc failed");
  if (rc == VSG_OK && !pair_supported(wt1, wt2, d1, L, (add0_bf16 ? 1 : 0) + (add1_bf16 ? 1 : 0), (out_raw_bf16 ? 1 : 0) + (out_act_bf16 ? 1 : 0))) rc = fail(VSG_EUNSUPPORTED, "shape not supported by the fused pair");
  if (rc == VSG_OK) {
    cudaMemset(err, 0, sizeof(int));
    EpiTC e;
    e.bias = wt2.bias;
    e.add0 = (const __nv_bfloat16*)add0_bf16; e.add1 = (const __nv_bfloat16*)add1_bf16;
    e.scale = scale; e.out_f32 = out_f32;
    e.out_raw = (__nv_bfloat16*)out_raw_bf16; e.out_act = (__nv_bfloat16*)out_act_bf16;
    TCOptions opt;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    rc = launch_pair_tc(&tmp, wt1, wt2, (const __nv_bfloat16*)xa_bf16, B, L, d1, e, opt, err, 0);
    if (rc == VSG_OK && g_debug_reps > 1) {
      cudaEventRecord(e0, 0);
      for (int r = 0; r < g_debug_reps && rc == VSG_OK; ++r)
        rc = launch_pair_tc(&tmp, wt1, wt2, (const __nv_bfloat16*)xa_bf16, B, L, d1, e, opt, err, 0);
      cudaEventRecord(e1, 0);
    }
    if (rc == VSG_OK) {
      cudaError_t ce = cudaDeviceSynchronize();
      if (ce != cudaSuccess) rc = fail(VSG_ECUDA, "pair_tc_kernel execution failed: %s", cudaGetErrorString(ce));
      else if (g_debug_reps > 1) { cudaEventElapsedTime(&g_debug_ms, e0, e1); g_debug_ms /= g_debug_reps; }
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
  }
  if (err) cudaFree(err);
  for (void* q : tmp.allocs) cudaFree(q);
  return rc;
}

// The fused pair as the decoder launches it, add0 activated or raw (tests only; allocates and synchronises).
// See include/visinger_b200.h.
extern "C" int vsg_debug_pair_tc(const VsgDebugPair* d, int32_t* image_out, int32_t device) {
  reset_launch_counts();
  if (!d || !d->xa || !d->w1 || !d->b1 || !d->w2 || !d->b2) return fail(VSG_EINVAL, "vsg_debug_pair_tc: null descriptor, input, weight or bias");
  if (d->B <= 0 || d->L <= 0 || d->C <= 0 || d->k <= 0 || d->d1 <= 0) return fail(VSG_EINVAL, "vsg_debug_pair_tc: bad shape");
  if (d->add0_is_act && !d->add0) return fail(VSG_EINVAL, "vsg_debug_pair_tc: add0_is_act without add0");
  const int C = d->C, k = d->k;
  DebugScope sc;
  VSG_TRY(sc.open(device));
  std::vector<float> W1(d->w1, d->w1 + (size_t)C * C * k), W2(d->w2, d->w2 + (size_t)C * C * k), B1(d->b1, d->b1 + C),
      B2(d->b2, d->b2 + C);
  ConvWTC wt1, wt2;
  VSG_TRY(pack_conv_tc(&sc.P, W1, B1, C, C, k, &wt1));
  VSG_TRY(pack_conv_tc(&sc.P, W2, B2, C, C, k, &wt2));
  if (!pair_supported(wt1, wt2, d->d1, d->L, (d->add0 ? 1 : 0) + (d->add1 ? 1 : 0), (d->out_raw ? 1 : 0) + (d->out_act ? 1 : 0)))
    return fail(VSG_EUNSUPPORTED, "vsg_debug_pair_tc: shape not supported by the fused pair");
  EpiTC e;
  e.bias = wt2.bias;
  e.add0 = (const __nv_bfloat16*)d->add0; e.add1 = (const __nv_bfloat16*)d->add1;
  e.add0_is_act = d->add0_is_act;
  e.scale = d->scale; e.out_f32 = d->out_f32;
  e.out_raw = (__nv_bfloat16*)d->out_raw; e.out_act = (__nv_bfloat16*)d->out_act;
  TCOptions opt;
  int img = -1;
  const int rc = launch_pair_tc(&sc.P, wt1, wt2, (const __nv_bfloat16*)d->xa, d->B, d->L, d->d1, e, opt, sc.err, 0, &img);
  if (image_out) *image_out = img;
  return sc.finish(rc);
}

// Per-layer parity hook for the whole-ResBlock1 kernel (tests and tuning only; allocates and synchronises).
//   xa: device bf16 [B, L, C] = leaky_relu(x); w: HOST fp32 [2 * n_pairs][C][C][k] in the order c1_0, c2_0, c1_1, ...;
//   b: HOST fp32 [2 * n_pairs][C]; out = (resblock1(x) [+ add1]) * scale.
extern "C" int vsg_debug_resblock_bf16(const void* xa_bf16, const float* w, const float* b, int32_t n_pairs,
                                       const int32_t* dilations, const void* add1_bf16, float scale, float* out_f32,
                                       void* out_raw_bf16, void* out_act_bf16, int32_t B, int32_t L, int32_t C, int32_t k,
                                       int32_t max_mb, int32_t sets, int32_t device) {
  reset_launch_counts();
  if (!xa_bf16 || !w || !b || !dilations || n_pairs < 1 || n_pairs > VSG_MAX_RESBLOCK_DILATIONS) return fail(VSG_EINVAL, "bad argument");
  VSG_CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  VSG_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  VsgPack tmp;
  tmp.device = device;
  tmp.sm_count = prop.multiProcessorCount;
  ResBlockPack rb;
  rb.kernel = k;
  rb.dilations.assign(dilations, dilations + n_pairs);
  rb.c1_tc.resize(n_pairs); rb.c2_tc.resize(n_pairs);
  rb.c1_rp.resize(n_pairs); rb.c2_rp.resize(n_pairs);
  rb.c1_x3.resize(n_pairs); rb.c2_x3.resize(n_pairs); rb.c1_rp_x3.resize(n_pairs); rb.c2_rp_x3.resize(n_pairs);
  const bool row_packed = (sets & 256) != 0;              // bit 8: the row-packed kernel (rp_tc.cuh); bit 9: no Toeplitz form
  const bool x3 = row_packed && (sets & 2048) != 0;       // bit 11: split-bf16 instantiation (two-plane tensors [B, L, 2 C])
  int rc = VSG_OK;
  const size_t wn = (size_t)C * C * k;
  std::vector<std::vector<float>> b2s;
  for (int q = 0; q < n_pairs; ++q) b2s.emplace_back(b + (2 * q + 1) * C, b + (2 * q + 2) * C);
  if (row_packed) rc = pack_resblock_bias_sums(&tmp, b2s, &rb);
  for (int q = 0; q < n_pairs && rc == VSG_OK; ++q) {
    std::vector<float> W1(w + (2 * q) * wn, w + (2 * q + 1) * wn), W2(w + (2 * q + 1) * wn, w + (2 * q + 2) * wn);
    std::vector<float> B1(b + (2 * q) * C, b + (2 * q + 1) * C), B2(b + (2 * q + 1) * C, b + (2 * q + 2) * C);
    rc = pack_conv_tc(&tmp, W1, B1, C, C, k, &rb.c1_tc[q]);
    if (rc == VSG_OK) rc = pack_conv_tc(&tmp, W2, B2, C, C, k, &rb.c2_tc[q]);
    if (rc == VSG_OK && row_packed && dilations[q] == 1) rc = pack_conv_rowpacked(&tmp, W1, C, k, &rb.c1_rp[q]);
    if (rc == VSG_OK && row_packed) rc = pack_conv_rowpacked(&tmp, W2, C, k, &rb.c2_rp[q]);
    if (x3) {
      if (rc == VSG_OK) rc = pack_conv_tc(&tmp, W1, B1, C, C, k, &rb.c1_x3[q], 2);
      if (rc == VSG_OK) rc = pack_conv_tc(&tmp, W2, B2, C, C, k, &rb.c2_x3[q], 2);
      if (rc == VSG_OK && dilations[q] == 1) rc = pack_conv_rowpacked(&tmp, W1, C, k, &rb.c1_rp_x3[q], 2);
      if (rc == VSG_OK) rc = pack_conv_rowpacked(&tmp, W2, C, k, &rb.c2_rp_x3[q], 2);
    }
  }
  int* err = nullptr;
  if (rc == VSG_OK && cudaMalloc(&err, sizeof(int)) != cudaSuccess) rc = fail(VSG_ECUDA, "cudaMalloc failed");
  if (rc == VSG_OK) {
    cudaMemset(err, 0, sizeof(int));
    TCOptions opt;
    opt.rb_max_mb = max_mb;
    if ((sets & 15) > 0) opt.rb_sets = sets & 15;       // bits 0-3: epilogue sets, bits 4-7: MMA issuer warps
    opt.rb_issuers = (sets >> 4) & 15;
    opt.rp_max_mb = max_mb;
    opt.rp_packed = (sets & 512) ? 0 : 1;
    opt.rp_spb2 = (sets & 1024) ? 1 : 0;              // bit 10: two epilogue warp sets per block, two blocks per set
    opt.rp_two_cta = (sets & 4096) ? 1 : 0;           // bit 12: the two-CTAs-per-SM form (8 epilogue warps, 2-block tiles)
    uint32_t* d_trace = nullptr;
    if (row_packed && getenv("VSG_RP_TRACE")) {
      cudaMalloc(&d_trace, 5 * 1024 * sizeof(uint32_t));
      cudaMemset(d_trace, 0, 5 * 1024 * sizeof(uint32_t));
      opt.rp_trace = d_trace;
    }
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    auto run = [&]() {
      if (row_packed)
        return launch_rp_tc(&tmp, rb, C, (const __nv_bfloat16*)xa_bf16, B, L, (const __nv_bfloat16*)add1_bf16,
                            (__nv_bfloat16*)out_raw_bf16, (__nv_bfloat16*)out_act_bf16, out_f32, scale, opt, err, 0, x3);
      return launch_rb_tc(&tmp, rb, C, (const __nv_bfloat16*)xa_bf16, B, L, (const __nv_bfloat16*)add1_bf16,
                          (__nv_bfloat16*)out_raw_bf16, (__nv_bfloat16*)out_act_bf16, out_f32, scale, opt, err, 0);
    };
    rc = run();
    if (rc == VSG_OK && g_debug_reps > 1) {
      cudaEventRecord(e0, 0);
      for (int r = 0; r < g_debug_reps && rc == VSG_OK; ++r) rc = run();
      cudaEventRecord(e1, 0);
    }
    if (rc == VSG_OK) {
      cudaError_t ce = cudaDeviceSynchronize();
      if (ce != cudaSuccess) rc = fail(VSG_ECUDA, "rb_tc_kernel execution failed: %s", cudaGetErrorString(ce));
      else if (g_debug_reps > 1) { cudaEventElapsedTime(&g_debug_ms, e0, e1); g_debug_ms /= g_debug_reps; }
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (d_trace) {   // issuer: (after waits, after commit) per block; epilogue sets: (before wait, after wait, before fence, after arrive)
      std::vector<uint32_t> h(5 * 1024);
      cudaMemcpy(h.data(), d_trace, h.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost);
      const uint32_t t0 = h[0];
      for (int r = 0; r < 5; ++r) {
        fprintf(stderr, "[rp trace] role %d:", r);
        for (int i = 0; i < 160 && h[r * 1024 + i]; ++i) fprintf(stderr, " %u", h[r * 1024 + i] - t0);
        fprintf(stderr, "\n");
      }
      cudaFree(d_trace);
    }
  }
  if (err) cudaFree(err);
  for (void* q : tmp.allocs) cudaFree(q);
  return rc;
}

// Per-kernel parity hook of the bf16 attention kernel (tests only; allocates and synchronises).  See include/visinger_b200.h.
extern "C" int vsg_debug_attention_bf16(const void* qkv_bf16, const float* mask, const float* ek, const float* ev, void* o_bf16,
                                        int32_t B, int32_t T, int32_t n_heads, int32_t dk, int32_t w, int32_t device) {
  reset_launch_counts();
  if (!qkv_bf16 || !mask || !ek || !ev || !o_bf16) return fail(VSG_EINVAL, "null pointer");
  if (B < 1 || T < 1 || n_heads < 1 || w < 0) return fail(VSG_EINVAL, "bad argument");
  VSG_CUDA_TRY(cudaSetDevice(device));
  int* err = nullptr;
  VSG_CUDA_TRY(cudaMalloc(&err, sizeof(int)));
  int rc = cudaMemset(err, 0, sizeof(int)) == cudaSuccess ? VSG_OK : fail(VSG_ECUDA, "cudaMemset failed");
  if (rc == VSG_OK)
    rc = attention_bf16(dk, (const __nv_bfloat16*)qkv_bf16, mask, ek, ev, (__nv_bfloat16*)o_bf16, B, n_heads, T, w, 0, nullptr,
                        err, 0);
  if (rc == VSG_OK) {
    int flag = 0;
    cudaError_t ce = cudaDeviceSynchronize();
    if (ce == cudaSuccess) ce = cudaMemcpy(&flag, err, sizeof(int), cudaMemcpyDeviceToHost);
    if (ce != cudaSuccess) rc = fail(VSG_ECUDA, "relenc_attention_tc_kernel execution failed: %s", cudaGetErrorString(ce));
    else if (flag) rc = fail(VSG_ECUDA, "relenc_attention_tc_kernel set its error flag (%d)", flag);
  }
  cudaFree(err);
  return rc;
}

// Per-kernel parity hook of the split-key attention path: the split launch plus the combine, at any T and a key chunk of
// key_chunk frames (a multiple of 128 up to 2048; 0 = 2048).  Tests only; allocates and synchronises.
extern "C" int vsg_debug_attention_split_bf16(const void* qkv_bf16, const float* mask, const float* ek, const float* ev,
                                              void* o_bf16, int32_t B, int32_t T, int32_t n_heads, int32_t dk, int32_t w,
                                              int32_t key_chunk, int32_t device) {
  reset_launch_counts();
  if (!qkv_bf16 || !mask || !ek || !ev || !o_bf16) return fail(VSG_EINVAL, "null pointer");
  if (B < 1 || T < 1 || n_heads < 1 || w < 0 || dk < 1) return fail(VSG_EINVAL, "bad argument");
  if (key_chunk == 0) key_chunk = 128 * tc::kAtMaxTiles;
  if (key_chunk < 0 || key_chunk % 128 || key_chunk > 128 * tc::kAtMaxTiles)
    return fail(VSG_EINVAL, "key chunk of %d frames (supported: a multiple of 128 up to %d, or 0)", key_chunk, 128 * tc::kAtMaxTiles);
  VSG_CUDA_TRY(cudaSetDevice(device));
  const int chunk_tiles = key_chunk / 128;
  int* err = nullptr;
  float* part = nullptr;
  VSG_CUDA_TRY(cudaMalloc(&err, sizeof(int)));
  int rc = cudaMalloc(&part, attention_split_floats(B, T, n_heads, dk, chunk_tiles) * sizeof(float)) == cudaSuccess
               ? VSG_OK : fail(VSG_ENOMEM, "cudaMalloc of the split-key partials failed");
  if (rc == VSG_OK && cudaMemset(err, 0, sizeof(int)) != cudaSuccess) rc = fail(VSG_ECUDA, "cudaMemset failed");
  if (rc == VSG_OK)
    rc = attention_bf16(dk, (const __nv_bfloat16*)qkv_bf16, mask, ek, ev, (__nv_bfloat16*)o_bf16, B, n_heads, T, w, chunk_tiles,
                        part, err, 0);
  if (rc == VSG_OK) {
    int flag = 0;
    cudaError_t ce = cudaDeviceSynchronize();
    if (ce == cudaSuccess) ce = cudaMemcpy(&flag, err, sizeof(int), cudaMemcpyDeviceToHost);
    if (ce != cudaSuccess) rc = fail(VSG_ECUDA, "split-key attention execution failed: %s", cudaGetErrorString(ce));
    else if (flag) rc = fail(VSG_ECUDA, "relenc_attention_tc_kernel set its error flag (%d)", flag);
  }
  if (part) cudaFree(part);
  cudaFree(err);
  return rc;
}

// Per-kernel parity hook of the bf16 encoder's fused LayerNorm -> condition -> mask step (tests only; synchronises).
extern "C" int vsg_debug_layernorm_bf16(void* x_bf16, const float* gamma, const float* beta, const float* g, int32_t g_t,
                                        const float* mask, float eps, int32_t B, int32_t T, int32_t C, int32_t device) {
  reset_launch_counts();
  if (!x_bf16 || !gamma || !beta || !mask) return fail(VSG_EINVAL, "null pointer");
  if (B < 1 || T < 1) return fail(VSG_EINVAL, "bad argument");
  if (C < 2 || C > 256 || (C & 1)) return fail(VSG_EUNSUPPORTED, "LayerNorm over %d channels (supported: even, <= 256)", C);
  VSG_CUDA_TRY(cudaSetDevice(device));
  const long long rows = (long long)B * T;
  relenc_layernorm_bf16_kernel<256><<<(unsigned)((rows + 7) / 8), 256>>>((__nv_bfloat16*)x_bf16, gamma, beta, g, g_t, mask, eps,
                                                                         C, T, rows);
  VSG_LAUNCH_CHECK("relenc_layernorm_bf16_kernel");
  const cudaError_t ce = cudaDeviceSynchronize();
  if (ce != cudaSuccess) return fail(VSG_ECUDA, "relenc_layernorm_bf16_kernel execution failed: %s", cudaGetErrorString(ce));
  return VSG_OK;
}

// Host-only: print the tile plan the launcher would choose for one convolution (tuning aid; no GPU needed).
extern "C" int vsg_debug_plan(int32_t Cin, int32_t Cout, int32_t k, int32_t dilation, int32_t B, int32_t L, int32_t n_adds,
                              int32_t n_outs, int32_t x3) {
  VsgPack tmp;
  ConvWTC wt;
  const int planes = x3 == 2 ? 3 : x3 ? 2 : 1;            // x3: 0 plain bf16, 1 two planes (split-bf16), 2 three planes (flow, fp32 tolerance)
  wt.Cin = Cin; wt.Cout = Cout; wt.CinT = planes * Cin; wt.CoutT = Cout; wt.ktaps = k; wt.has_tmap = true;
  wt.x3 = planes == 2; wt.planes = planes;
  static __nv_bfloat16 dummy, dummy_in;                    // (a k > 1 convolution must not alias its input)
  EpiTC e;
  if (n_adds > 0) e.add0 = &dummy;
  if (n_adds > 1) e.add1 = &dummy;
  if (n_outs > 0) e.out_act = &dummy;
  if (n_outs > 1) e.out_raw = &dummy;
  TCOptions opt = g_default_opts;
  opt.plan_only = 1;
  return launch_conv_tc(&tmp, wt, &dummy_in, B, L, -((k - 1) * dilation / 2), dilation, L, 1, 0, L, e, opt, nullptr, 0);
}

// Host-only: the tile plan of the fused ResBlock1 pair (pair_tc.cuh) for one shape; no GPU needed.
//   out[3]: 128-row blocks per tile, valid output rows per tile, tiles per utterance
// Returns VSG_EUNSUPPORTED when the pair kernel does not take the shape (the decoder then runs the two convolutions apart).
extern "C" int vsg_debug_pair_plan(int32_t C, int32_t k, int32_t d1, int32_t L, int32_t n_adds, int32_t n_outs, int32_t* out) {
  if (!out || C <= 0 || k <= 0 || d1 <= 0 || L <= 0 || n_adds < 0 || n_adds > 2 || n_outs < 0 || n_outs > 2)
    return fail(VSG_EINVAL, "bad argument");
  ConvWTC w;                                  // what pack_conv_tc would record for this shape
  w.Cin = C; w.Cout = C; w.CinT = C; w.CoutT = C; w.ktaps = k; w.has_tmap = true; w.x3 = false; w.planes = 1;
  if (!pair_supported(w, w, d1, L, n_adds, n_outs)) return fail(VSG_EUNSUPPORTED, "shape not supported by the fused pair");
  const int V = pair_valid_rows(C, k);
  out[0] = pair_mb(C); out[1] = V; out[2] = (L + V - 1) / V;
  return VSG_OK;
}

// Host-only: the tile plan of the row-packed whole-ResBlock1 kernel (rp_tc.cuh) for one resblock shape; no GPU needed.
//   variant: 0 plain bf16, 1 split-bf16 (bf16x3 mode), 2 plain bf16 as two CTAs per SM
//   out[8]: mb, H, V, ring stages, dynamic shared memory (bytes), packed mask, tiles per utterance, accumulator columns
// Returns VSG_EUNSUPPORTED when the kernel does not take the shape (the caller then runs the per-convolution kernels).
extern "C" int vsg_debug_rp_plan(int32_t C, int32_t k, int32_t n_pairs, const int32_t* dilations, int32_t L, int32_t variant,
                                 int32_t* out) {
  if (!dilations || !out || n_pairs < 1 || n_pairs > VSG_MAX_RESBLOCK_DILATIONS) return fail(VSG_EINVAL, "bad argument");
  const bool x3 = variant == 1;
  ResBlockPack rb;
  rb.kernel = k;
  rb.dilations.assign(dilations, dilations + n_pairs);
  ConvWTC w;                                  // what pack_conv_tc / pack_conv_rowpacked would record for this shape
  w.Cin = C; w.Cout = C; w.CinT = (x3 ? 2 : 1) * C; w.CoutT = C; w.ktaps = k; w.has_tmap = true; w.x3 = x3; w.planes = x3 ? 2 : 1;
  ConvWTC wp = w;
  wp.has_tmap = (C == 16 || C == 32) && (k % 2 == 1);
  rb.c1_tc.assign(n_pairs, w); rb.c2_tc.assign(n_pairs, w);
  rb.c1_x3.assign(n_pairs, w); rb.c2_x3.assign(n_pairs, w);
  rb.c1_rp.assign(n_pairs, wp); rb.c2_rp.assign(n_pairs, wp);
  rb.c1_rp_x3.assign(n_pairs, wp); rb.c2_rp_x3.assign(n_pairs, wp);
  if (x3) for (auto* v : {&rb.c1_tc, &rb.c2_tc}) for (auto& e : *v) { e.x3 = false; e.planes = 1; e.CinT = C; }
  rb.c2_bsum.assign(n_pairs, nullptr);
  TCOptions opt = g_default_opts;
  opt.rp_two_cta = variant == 2 ? 1 : 0;
  RpPlan pl;
  if (!rp_plan(rb, C, L, opt, &pl, x3)) return fail(VSG_EUNSUPPORTED, "resblock shape not supported by the row-packed kernel");
  uint32_t tmem = 32;
  while (tmem < (uint32_t)(2 * pl.mb * 64)) tmem <<= 1;
  out[0] = pl.mb; out[1] = pl.H; out[2] = pl.V; out[3] = pl.n_wst; out[4] = (int32_t)pl.smem; out[5] = (int32_t)pl.packed_mask;
  out[6] = (L + pl.V - 1) / pl.V; out[7] = (int32_t)tmem;
  return VSG_OK;
}

// Select the default A-operand feeding mode of the tensor-core convolutions (process-wide; tests and tuning).
extern "C" int vsg_set_tc_options(int32_t halo_mode, int32_t w_resident, int32_t l2_tensor_mb, int32_t min_tiles) {
  g_default_opts.halo_mode = halo_mode & 1;
  g_default_opts.w_resident = w_resident;
  g_default_opts.max_mb = ((halo_mode >> 4) & 15) ? ((halo_mode >> 4) & 15) : 4;   // bits 4..7: cap on blocks per tile
  g_default_opts.use_pdl = (halo_mode & 256) ? 0 : 1;                               // bit 8: disable dependent launch
  g_default_opts.fuse_pairs = (halo_mode & 512) ? 0 : 1;                            // bit 9: disable fused resblock pairs
  g_default_opts.merge_ups = (halo_mode & 1024) ? 0 : 1;                            // bit 10: one launch per polyphase
  g_default_opts.split_n = (halo_mode & 2048) ? 0 : 1;                              // bit 11: never split N = 256 tiles
  g_default_opts.single_stream = (halo_mode & 4096) ? 0 : 1;                        // bit 12: store raw + activated copies
  g_default_opts.epi_sigs = (halo_mode & 8192) ? 0 : (halo_mode & (1 << 27)) ? 1 : 2; // bit 13: generic epilogue kernels only; bit 27: no SUM / FINAL images
  g_default_opts.chain_streams = (halo_mode & 16384) ? 0 : 1;                       // bit 14: resblock chains on one stream
  g_default_opts.epi_sets = (halo_mode & 8192) ? 1 : 2;                             // bit 13: one set of epilogue warps
  g_default_opts.fuse_rb = (halo_mode & 32768) ? 1 : 0;                             // bit 15: whole-resblock kernel
  g_default_opts.rb_max_mb = (halo_mode >> 16) & 31;                                // bits 16-20: cap on blocks per resblock tile
  g_default_opts.rb_sets = ((halo_mode >> 21) & 7) ? ((halo_mode >> 21) & 7) : 4;   // bits 21-23: resblock epilogue warp sets
  g_default_opts.fuse_rp = (halo_mode & (1 << 24)) ? 0 : 1;                         // bit 24: no row-packed resblock kernel
  g_default_opts.rp_max_c = (halo_mode & (1 << 25)) ? 64 : 32;                      // bit 25: row-packed kernel at C = 64 too
  g_default_opts.rp_packed = (halo_mode & (1 << 26)) ? 0 : 1;                       // bit 26: no block-Toeplitz form
  g_default_opts.rp_two_cta = (halo_mode & 4) ? 1 : 0;                              // bit 2: row-packed kernel as two CTAs per SM
  g_default_opts.rp_x3 = (halo_mode & 2) ? 0 : 1;                                   // bit 1: bf16x3 mode without the row-packed resblock kernel
  g_default_opts.rp_spb2 = (halo_mode & (1 << 30)) ? 1 : 0;                         // bit 30: row-packed kernel, two epilogue sets per block
  g_default_opts.flow_merge = ((uint32_t)halo_mode & (1u << 31)) ? 0 : 1;           // bit 31: flow with separate res / skip / cond launches
  g_default_opts.conv_post = (halo_mode >> 28) & 3;                                 // bits 28-29: conv_post on CUDA cores (1 / 2)
  if (l2_tensor_mb >= 0) g_l2_tensor_mb = l2_tensor_mb;
  if (min_tiles > 0) g_min_tiles = min_tiles;
  return VSG_OK;
}
