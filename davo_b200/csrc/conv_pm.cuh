// Implicit-GEMM convolution on the 5th-gen tensor cores (tcgen05, TF32 in /
// fp32 accumulate in TMEM), operands fed by TMA.  One kernel serves every conv
// of the PoseNN stack (reference nets/posenn.py:211-215, 238-240):
//
//   out[pixel, n] = act( bias[n] + sum_{tap} A_tap[pixel, 0:32] . B_tap[n, 0:32] )
//
// * M tile = 128 output pixels = a 16 (rows) x 8 (cols) block of one frame pair.
// * A "tap" is one 32-float (128 B) slab of the reduction axis: a filter tap (or,
//   for the thin strided layers, 2 or 4 horizontally adjacent taps) x 32 / 16 / 8
//   input channels.
// * The A operand is never gathered per tap.  A PATCH -- the tile's input halo,
//   {32 ch, Wp cols, 1, Hp rows, 1} of the NHWC activation -- is loaded ONCE by
//   a 5-D TMA box placed with signed coordinates, so TF-'SAME' padding (asymmetric
//   included) is TMA's out-of-bounds zero fill.  The box lands as Hp*Wp rows of
//   128 B with SWIZZLE_128B.  Every tap of the patch is then just a different
//   UMMA descriptor: start address = patch + (row*Wp + col)*128 B, 8-row groups
//   SBO = Wp*128 B apart.  (The hardware swizzle is a function of the absolute
//   shared-memory address, so a row-shifted window needs no re-layout -- measured,
//   tools/experiments/desc_shift.cu.)  Dilation is only a tap offset: no im2col
//   buffer, no space-to-batch, each input byte crosses L2->SM once per tile.
// * Stride-2 layers view the input as [N][H/2][2][W/2][2*C]: a tap is a unit-stride
//   window at one (row parity, column parity) of that view; one patch per parity.
// * B (weights, pre-packed [tap][Cout][32], TF32-rounded) is either streamed
//   through a ring (one 2-D TMA box per tap) or, for the thin layers, loaded once
//   and kept resident in shared memory for the CTA's whole life.
//
// * Column-widened form (WIDE; the thin stride-2 layers cnv1, cnv2).  One tcgen05.mma of
//   M=128, K=8 costs 53.8 cycles however small N is (64 at N=128;
//   tools/experiments/mma_floor.cu), so a 16-channel layer with pixels on M is bound by the
//   NUMBER of MMAs.  Here one M row is a run of G horizontally adjacent output pixels of one
//   image row and N = G x Cout = 128 holds all of them.  A slab is S input pixels x C channels
//   (32 floats: C = 16, S = 2 for cnv2; the 8-channel packed input gives cnv1 S = 4).  Slab c
//   of a run feeds output pixel g through the filter columns tx = 2d + wp + pad_l with
//   d = (S/2)c - g, so its weight operand is a WINDOW of one resident block
//   [W[d_max]; ...; W[d_min]] per filter row and its result a window of the accumulator
//   (per-tap N, first column and first weight row: davo_capi.cu, plan_layer_wide).  Every slab
//   position c is its own patch {32 floats at 32*(c mod slabs_per_run), tile_w runs, 1 parity,
//   Hp rows, 1} of the view [N][H/2][2][W/2G][2G*C]; a tile is tile_h rows x tile_w runs with
//   tile_w == Wp, so its 128 M rows are 128 consecutive 128-B slabs.  cnv1: 172 MMAs per 1024
//   pixels instead of 896.
//
// Warp roles (224 threads): warp 0 patch (A) TMA producer, warp 6 weight (B) TMA producer,
// warp 1 TMEM owner + MMA issue (all 32 lanes run the loop so that every operand lives on the
// uniform datapath; elect.sync picks the issuing lane), warps 2-5 epilogue: TMEM -> registers ->
// bias/ReLU/round -> a per-warp swizzled staging buffer -> one TMA tile store per 32x32 block
// (or the spatial-sum epilogue of cnv7).  Accumulators are double-buffered in TMEM so the
// epilogue of tile i overlaps the main loop of tile i+1.  Persistent CTAs walk tiles
// round-robin.
#pragma once
#include "conv_common.cuh"
#include "frontend.cuh"

namespace davo {
namespace pm {

constexpr int kTileM = 128;
constexpr int kTileH = 16;
constexpr int kEpiStageBytes = 4 * 2 * 4096;        // 4 epilogue warps x 2 buffers x (32 pixels x 128 B)
constexpr int kBiasSmemBytes = 2048;                // up to 512 bias floats
#ifndef DAVO_FUSED_WARPS
#define DAVO_FUSED_WARPS 8
#endif
constexpr int kFusedWarps = DAVO_FUSED_WARPS;       // FUSED: warps 7.. build the patches from the raw inputs
constexpr int kFusedThreads = kFusedWarps * 32;
constexpr int kFusedItems = kFusedWarps >= 16 ? 2 : kFusedWarps >= 12 ? 3 : 4;      // slabs of a half a producer thread builds at most

// FUSED (cnv1 on the 8-channel packed input): what the front end would have written to memory is built in shared
// memory instead.  The patches of a tile come in two halves, one per row parity; for a half the producers
//   A. copy the raw inputs of its rows -- Hp rows x raw_px pixels: flow (float2), the target's and the source's image
//      bytes, the labels as bytes -- into a staging area with coalesced copies (a warp reads whole row segments), then
//   B. build the half's patches one after the other, in the order the MMA warp consumes them: a thread takes a slab
//      (4 pixels x 8 channels), reads its 4 pixels from the staging area, applies pack8_quad (frontend.cuh: the same
//      function pack8_kernel stores through, so the operand bits are the same) and writes the 128 B where TMA would
//      have put them (16-B chunks XOR-swizzled by row & 7), fences them for the async proxy and arrives on the patch's
//      barrier (one arrival per slab).
// There are two staging areas: the copies of step c + 1 (cp.async, plus the float labels held in registers) are issued
// before the patches of step c are built and have that whole step to land.  To make room the fused kernel keeps one
// epilogue buffer per warp instead of two and a ring of three patches.  Experiment, off by default: same bits as
// pack8_kernel + cnv1, even in time (DESIGN.md 4.2, profiles/r2_experiment_fused_front_v2.log).
struct FusedGeo {
  int raw_px;          // pixels per staged row (multiple of 4)
  int flow_pitch;      // float4 per staged flow row: raw_px / 2 + 1
  int x_lo;            // first staged pixel relative to the tile's first input column (2 * G * w0)
  int half_patches;    // patches per row parity; patches [0, half) share one parity and dh, [half, 2 half) the other
  int off_tgt, off_src, off_lab_s, off_lab_t;      // byte offsets in the staging area (flow first, at 0)
  int raw_off;         // first staging area: bytes from the 1024-aligned start of dynamic shared memory
  int raw_bytes;       // size of one staging area; the second follows the first
};

struct ConvParams {
  int num_tiles;        // pairs * groups * tiles_h * tiles_w
  int tiles_w, tiles_h, groups;
  int Hout, Wout;
  int out_stride;       // floats per output pixel (all groups)
  int cin_group_off;    // inner-coordinate offset of group g = g * cin_group_off
  int n_patches, n_taps;          // per tile
  int patch_w;                    // Wp
  int patch_bytes;                // Hp * Wp * 128 (what TMA delivers)
  int patch_stage_bytes;          // rounded up to 1024
  int p_stages, b_stages;         // ring depths (b_stages unused when B is resident)
  // WIDE only
  int tile_h, tile_w;             // tile = tile_h output rows x tile_w runs (tile_h * tile_w = 128)
  int run_px;                     // G: output pixels per run (per M row)
  int b_boxes, b_box_rows;        // resident weights: one TMA box of b_box_rows rows per filter row
  int raw;                        // store epilogue: 1 = plain fp32 sums, no relu, no rounding (-batch_norm: bn.cuh finishes the layer)
  float* out;           // EPI_STORE: [pairs][Hout][Wout][out_stride]
  const float* bias;    // [groups * BN]
  float* sum_out;       // EPI_SUM:   [pairs][groups][tiles_h*tiles_w][4][BN]
  FusedGeo fg;          // FUSED only
  FrontParams front;    // FUSED only: the inputs and variant switches of the attention front end
  PatchDesc patches[kMaxPatches];
  TapDesc taps[kMaxTaps];
};

template <int BN>
struct ConvCfg {
  static constexpr int kBBytes = BN * kSlabBytes;
  static constexpr int kAccStride = BN < 32 ? 32 : BN;             // TMEM columns per accumulator
  static constexpr int kTmemCols = 2 * kAccStride;                 // power of two for BN in {16..256}
};

template <int BN, int EPI, bool B_RESIDENT, bool WIDE = false, bool FUSED = false>
__global__ void __launch_bounds__(kConvThreads + (FUSED ? kFusedThreads : 0), 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmO, const __grid_constant__ ConvParams p) {
  using Cfg = ConvCfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B operands: keep every stage base 1024-B aligned.
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~uintptr_t(1023));
  const int PS = p.p_stages;
  static_assert(!WIDE || (B_RESIDENT && EPI == EPI_STORE_RELU && BN >= 32), "WIDE: resident weights, store epilogue");
  static_assert(!FUSED || WIDE, "the fused front end feeds the column-widened cnv1 plan");
  const int BS = B_RESIDENT ? p.n_taps * p.groups : p.b_stages;   // resident: every slab has a home
  const int b_bytes = WIDE ? p.b_boxes * p.b_box_rows * kSlabBytes : BS * Cfg::kBBytes;
  const int TH = WIDE ? p.tile_h : kTileH, TW = WIDE ? p.tile_w : kTileW;
  uint8_t* smem_p = smem;
  uint8_t* smem_b = smem + PS * p.patch_stage_bytes;
  uint8_t* epi_stage = smem_b + b_bytes;                           // 1024-B aligned (TMA store, 128-B swizzle)
  constexpr int kEpiBytes = FUSED ? kEpiStageBytes / 2 : kEpiStageBytes;      // FUSED: one staging buffer per epilogue warp
  uint64_t* bars = reinterpret_cast<uint64_t*>(epi_stage + kEpiBytes);
  uint64_t* p_full = bars;                        // [kMaxStages] TMA -> MMA
  uint64_t* p_empty = bars + kMaxStages;          // [kMaxStages] MMA -> TMA
  uint64_t* b_full = bars + 2 * kMaxStages;       // [kMaxStages] (resident: [0] only)
  uint64_t* b_empty = bars + 3 * kMaxStages;      // [kMaxStages]
  uint64_t* acc_full = bars + 4 * kMaxStages;     // [2] MMA -> epilogue
  uint64_t* acc_empty = acc_full + 2;             // [2] epilogue -> MMA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  float* bias_s = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + kBarrierBytes);

  pdl_launch_dependents();
  const EpiAct ea = epi_act(p.raw);
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);   // known warp-uniform to the compiler
  const int lane = threadIdx.x & 31;
#ifdef DAVO_TIMING
  long long tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const long long t_cta0 = clock64();
#endif

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if constexpr (EPI == EPI_STORE_RELU) tma_prefetch_desc(&tmO);
    for (int i = 0; i < kMaxStages; ++i) {
      mbar_init(&p_full[i], FUSED ? (uint32_t)(p.patch_bytes / kSlabBytes) : 1u);   // FUSED: one arrival per slab
      mbar_init(&p_empty[i], 1);
      mbar_init(&b_full[i], 1);
      mbar_init(&b_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], 4);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, Cfg::kTmemCols);
  for (int i = threadIdx.x; i < p.groups * BN; i += blockDim.x) bias_s[i] = p.bias[i];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int tiles_per_img = p.tiles_h * p.tiles_w;
  const int tiles_per_pair = tiles_per_img * p.groups;

  if (FUSED && warp >= 7) {
    // ------------------------------------- patch producers: fused front end --
    const FrontParams& f = p.front;
    const FusedGeo& fg = p.fg;
    const int ptid = (int)threadIdx.x - kConvThreads;
    uint8_t* raw0 = smem + fg.raw_off;                            // two staging areas, fg.raw_bytes apart: step c uses area c & 1
    float* wtab0 = bias_s + 256;                                  // class weights, two sets (by tile parity) of [32 source | 32 target]
    const int spp = p.patch_bytes / kSlabBytes;                   // slabs per patch: Hp x tile_w
    const int Hp = spp / p.tile_w;
    const int NF = fg.raw_px / 2, NT = fg.raw_px * 3 / 4, NL = fg.raw_px / 4;     // float4 / u32 / u32 per staged row
    const int NFP = fg.flow_pitch;                                // float4 per staged flow row (NF + 1: rows start in different banks)
    const bool lab_s = f.att_src != 0, lab_t = lab_s && !f.att_tgt_ones, use_flow = f.in_mode == 1;
    const int hw = f.H * f.W;
    // This thread's slabs of a half: the same positions in every tile (kFusedItems of them at most; step B below)
    int it_pos[kFusedItems], it_xr[kFusedItems];                  // within | patch-in-half << 16 (-1: none); staged column per half
#pragma unroll
    for (int t = 0; t < kFusedItems; ++t) {
      const int i = ptid + t * kFusedThreads;
      it_pos[t] = -1; it_xr[t] = 0;
      if (i < fg.half_patches * spp) {
        const int qp = i / spp, within = i - qp * spp, j = within % p.tile_w;
        it_pos[t] = within | (qp << 16);
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const PatchDesc d = p.patches[half * fg.half_patches + qp];
          it_xr[t] |= (2 * p.run_px * (j + d.dw) + (d.c >> 5) * 4 - fg.x_lo) << (16 * half);
        }
      }
    }
    // A step is one half of one tile: step c = half (c & 1) of this CTA's tile number (c >> 1).
    struct Step { int ok, n, b, k, y0, X0; };
    auto step_of = [&](int c) {
      Step s;
      const int tile = (int)blockIdx.x + (c >> 1) * (int)gridDim.x;
      s.ok = tile < p.num_tiles;
      s.n = s.b = s.k = s.y0 = s.X0 = 0;
      if (s.ok) {
        s.n = tile / tiles_per_pair;
        const int r = tile - s.n * tiles_per_pair;
        const PatchDesc d = p.patches[(c & 1) * fg.half_patches];
        s.y0 = 2 * ((r / p.tiles_w) * TH + d.dh) + d.par;         // input row of staged row 0; staged row rr is y0 + 2 rr
        s.X0 = 2 * p.run_px * ((r % p.tiles_w) * TW) + fg.x_lo;    // first staged input column
        pair_of_slot(f.pair_mode, f.pair0 + s.n, &s.b, &s.k);
      }
      return s;
    };
    // float labels travel through registers (they are narrowed to bytes on the way): loaded by stage_issue, stored by
    // stage_finish after the patches of the step before have been built
    constexpr int kLabRegs = 3;
    float4 lab_v[kLabRegs];
    uint32_t lab_mask = 0;
    auto narrow4 = [](const float4 v) {
      const int l4[4] = {label_of(v.x), label_of(v.y), label_of(v.z), label_of(v.w)};
      uint32_t w4 = 0;
#pragma unroll
      for (int i = 0; i < 4; ++i) w4 |= (uint32_t)((l4[i] >= 0 && l4[i] < kNumClasses) ? l4[i] : 255) << (8 * i);
      return w4;
    };
    // ---- A: the raw inputs of a step, on their way into its staging area ----
    // The flow and the image bytes (and byte labels) go global -> shared asynchronously (cp.async: no registers in between,
    // every copy of the half in flight at once).  A thread keeps its column and walks down the rows: no division in the loops.
    auto stage_issue = [&](const Step& s, int c) {
      uint8_t* raw = raw0 + (c & 1) * fg.raw_bytes;
      const uint32_t raw_u = smem_u32(raw);
      const int b = s.b, k = s.k, y0 = s.y0, X0 = s.X0;
      const size_t seg_src = frame_plane(f.in, b, k == 0 ? 0 : 2, hw), seg_tgt = frame_plane(f.in, b, 1, hw);
      if ((c & 1) == 0 && ptid < 2 * kNumClasses) {               // the tile's class weights
        const bool se = f.att_src == 1 || f.att_src >= 3;
        const int fr = ptid / kNumClasses, cl = ptid - fr * kNumClasses;
        wtab0[((c >> 1) & 1) * 64 + fr * 32 + cl] =
            (se && (fr == 0 || !f.att_tgt_ones)) ? __ldcg(f.att_w + ((size_t)s.n * kAttFrames + fr) * kAttStride + cl)
            : f.att_src == 2 ? f.static_w[cl] : 1.0f;
      }
      const bool flow_plain = use_flow && !f.flow_f16 && b >= f.in.n_flow16;    // float32 flow used as it is
      if (flow_plain) {
        const int RF = kFusedThreads / NF, r0 = ptid / NF, e = ptid - r0 * NF, x = X0 + 2 * e;      // two pixels of flow
        if (r0 < RF && x >= 0 && x < f.W) {
          const float* fsrc = flow_plane(f.in, b, k) + (size_t)x * 2;
          for (int rr = r0; rr < Hp; rr += RF) {
            const int y = y0 + 2 * rr;
            if (y >= 0 && y < f.H) cp_async_16(raw_u + (rr * NFP + e) * 16, fsrc + (size_t)y * f.W * 2);
          }
        }
      }
      {
        const int RI = kFusedThreads / (2 * NT), r0 = ptid / (2 * NT), e = ptid - r0 * 2 * NT;
        const int fr = e >= NT, wd = e - fr * NT;                        // one 32-bit word of the target's / the source's image bytes
        const int x = X0 + (wd / 3) * 4;                                 // the quad the word belongs to
        if (r0 < RI && x >= 0 && x < f.W) {
          // (16-byte copies of the aligned middle of a row were tried: slower than word copies, 0.371 against 0.348 ms)
          const uint8_t* isrc = frame_img(f.in, b, fr ? (k == 0 ? 0 : 2) : 1) + (size_t)X0 * 3 + wd * 4;
          const uint32_t dst0 = raw_u + (fr ? fg.off_src : fg.off_tgt) + wd * 4;
          for (int rr = r0; rr < Hp; rr += RI) {
            const int y = y0 + 2 * rr;
            if (y >= 0 && y < f.H) cp_async_4(dst0 + rr * NT * 4, isrc + (size_t)y * f.in.img_row);
          }
        }
      }
      if (use_flow && !flow_plain) {                     // binary16 flow (opt-in) / half planes from the host: through flow2_at
        constexpr int U = 6;
        for (int i0 = ptid; i0 < Hp * NF; i0 += kFusedThreads * U) {
          float4 v[U];
          int dst[U];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int idx = i0 + u * kFusedThreads, rr = idx / NF, e = idx - rr * NF;
            const int y = y0 + 2 * rr, x = X0 + 2 * e;
            dst[u] = (idx < Hp * NF && y >= 0 && y < f.H && x >= 0 && x < f.W) ? rr * NFP + e : -1;
            if (dst[u] >= 0) v[u] = flow2_at(f, b, k, y * f.W + x, hw);
          }
#pragma unroll
          for (int u = 0; u < U; ++u)
            if (dst[u] >= 0) *reinterpret_cast<float4*>(raw + (size_t)dst[u] * 16) = v[u];
        }
      }
      lab_mask = 0;
      if (lab_s) {                                                       // four labels -> four bytes (255: no class)
        const int per_row = lab_t ? 2 * NL : NL, RL = kFusedThreads / per_row, r0 = ptid / per_row, e = ptid - r0 * per_row;
        const int fr = e >= NL, qd = e - fr * NL, x = X0 + 4 * qd;
        if (r0 < RL && x >= 0 && x < f.W) {
          const size_t plane = (fr ? seg_tgt : seg_src) + x;
          const int dst0 = (fr ? fg.off_lab_t : fg.off_lab_s) + qd * 4;
          if (f.in.seg8) {
            for (int rr = r0; rr < Hp; rr += RL) {
              const int y = y0 + 2 * rr;
              if (y >= 0 && y < f.H) cp_async_4(raw_u + dst0 + rr * NL * 4, f.in.seg8 + plane + (size_t)y * f.W);
            }
          } else {
#pragma unroll
            for (int u = 0; u < kLabRegs; ++u) {                         // the loads only: their values are first used in stage_finish
              const int rr = r0 + u * RL, y = y0 + 2 * rr;
              if (rr < Hp && y >= 0 && y < f.H) {
                lab_v[u] = __ldg(reinterpret_cast<const float4*>(f.in.seg + plane + (size_t)y * f.W));
                lab_mask |= 1u << u;
              }
            }
            for (int rr = r0 + kLabRegs * RL; rr < Hp; rr += RL) {        // more rows than registers (target labels too): on the spot
              const int y = y0 + 2 * rr;
              if (y >= 0 && y < f.H)
                *reinterpret_cast<uint32_t*>(raw + dst0 + rr * NL * 4) = narrow4(__ldg(reinterpret_cast<const float4*>(f.in.seg + plane + (size_t)y * f.W)));
            }
          }
        }
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto stage_finish = [&](int c) {                                     // the labels that waited in registers, narrowed to bytes
      if (lab_mask == 0) return;
      uint8_t* raw = raw0 + (c & 1) * fg.raw_bytes;
      const int per_row = lab_t ? 2 * NL : NL, RL = kFusedThreads / per_row, r0 = ptid / per_row, e = ptid - r0 * per_row;
      const int fr = e >= NL, qd = e - fr * NL;
#pragma unroll
      for (int u = 0; u < kLabRegs; ++u)
        if (lab_mask & (1u << u))
          *reinterpret_cast<uint32_t*>(raw + (fr ? fg.off_lab_t : fg.off_lab_s) + ((r0 + u * RL) * NL + qd) * 4) = narrow4(lab_v[u]);
    };
    int ring_stage0 = 0;                                          // ring stage and use count of the current half's first patch
    uint32_t ring_use0 = 0;
    pdl_wait();                     // the class weights come from the SE kernel before this one
    Step cur = step_of(0);
    if (cur.ok) { stage_issue(cur, 0); stage_finish(0); }
    for (int c = 0; cur.ok; ++c) {
      // The copies of the NEXT step start now, into the other staging area, and fly while this step's patches are built
      const Step nxt = step_of(c + 1);
      if (nxt.ok) stage_issue(nxt, c + 1);
      else asm volatile("cp.async.commit_group;" ::: "memory");
      asm volatile("cp.async.wait_group 1;" ::: "memory");          // all but the newest group: this step's copies have landed
      asm volatile("bar.sync 1, %0;" ::"n"(kFusedThreads) : "memory");       // ... for every producer thread
      // ---- B: the patches of this half, in ring order ----
      const uint8_t* raw = raw0 + (c & 1) * fg.raw_bytes;
      const float* wtab = wtab0 + ((c >> 1) & 1) * 64;
      const int half = c & 1, y0 = cur.y0, X0 = cur.X0;
#pragma unroll
      for (int t = 0; t < kFusedItems; ++t) {
        if (it_pos[t] < 0) continue;
        const int qp = it_pos[t] >> 16, within = it_pos[t] & 0xFFFF;
        const int rr = within / p.tile_w;
        const int xr = (it_xr[t] >> (16 * half)) & 0xFFFF;                        // staged column of the slab's first pixel
        const int y = y0 + 2 * rr, x = X0 + xr;
        float4 q[8];
#pragma unroll
        for (int cc = 0; cc < 8; ++cc) q[cc] = make_float4(0.f, 0.f, 0.f, 0.f);            // 'SAME' padding
        if (y >= 0 && y < f.H && x >= 0 && x < f.W) {
          const int qd = xr >> 2;
          const uint32_t* tw = reinterpret_cast<const uint32_t*>(raw + fg.off_tgt + ((size_t)rr * NT + 3 * qd) * 4);
          const uint32_t* sw = reinterpret_cast<const uint32_t*>(raw + fg.off_src + ((size_t)rr * NT + 3 * qd) * 4);
          int ls[4] = {-1, -1, -1, -1}, lt[4] = {-1, -1, -1, -1};
          if (lab_s) {
            const uint32_t w4 = *reinterpret_cast<const uint32_t*>(raw + fg.off_lab_s + ((size_t)rr * NL + qd) * 4);
            ls[0] = w4 & 255u; ls[1] = (w4 >> 8) & 255u; ls[2] = (w4 >> 16) & 255u; ls[3] = w4 >> 24;
          }
          if (lab_t) {
            const uint32_t w4 = *reinterpret_cast<const uint32_t*>(raw + fg.off_lab_t + ((size_t)rr * NL + qd) * 4);
            lt[0] = w4 & 255u; lt[1] = (w4 >> 8) & 255u; lt[2] = (w4 >> 16) & 255u; lt[3] = w4 >> 24;
          }
          float4 f0 = make_float4(0.f, 0.f, 0.f, 0.f), f1 = f0;
          if (use_flow) {
            f0 = *reinterpret_cast<const float4*>(raw + ((size_t)rr * NFP + 2 * qd) * 16);
            f1 = *reinterpret_cast<const float4*>(raw + ((size_t)rr * NFP + 2 * qd + 1) * 16);
          }
          pack8_quad(f, wtab, wtab + 32, tw[0], tw[1], tw[2], sw[0], sw[1], sw[2], ls, lt, f0, f1, q);
        }
        int stage = ring_stage0 + qp;                                // the patch's place in the ring's life
        uint32_t use = ring_use0;
        while (stage >= PS) { stage -= PS; ++use; }
        mbar_wait(&p_empty[stage], (use & 1u) ^ 1u);
        const uint32_t row = smem_u32(smem_p + stage * p.patch_stage_bytes) + (uint32_t)within * kSlabBytes;
#pragma unroll
        for (int cc = 0; cc < 8; ++cc) sts_v4(row + ((cc ^ (within & 7)) << 4), q[cc]);
        fence_proxy_async_smem();
        mbar_arrive(&p_full[stage]);
      }
      ring_stage0 += fg.half_patches;
      while (ring_stage0 >= PS) { ring_stage0 -= PS; ++ring_use0; }
      if (nxt.ok) stage_finish(c + 1);
      asm volatile("bar.sync 1, %0;" ::"n"(kFusedThreads) : "memory");       // this step's staging area has been read by everyone
      cur = nxt;
    }
  } else if (warp == 0) {
    // ------------------------------------------------- patch (A) producer --
    if (lane == 0 && !FUSED) {
      pdl_wait();                 // the activations this layer reads are the previous kernel's output
      int ps = 0;
      uint32_t pphase = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        const int n = tile / tiles_per_pair;
        int r = tile - n * tiles_per_pair;
        const int g = r / tiles_per_img;
        r -= g * tiles_per_img;
        const int h0 = (r / p.tiles_w) * TH;
        const int w0 = (r % p.tiles_w) * TW;
        for (int pi = 0; pi < p.n_patches; ++pi) {
          const PatchDesc d = p.patches[pi];
          TWAIT(0, mbar_wait(&p_empty[ps], pphase ^ 1));
          mbar_expect_tx(&p_full[ps], p.patch_bytes);
          tma_load_5d(smem_p + ps * p.patch_stage_bytes, &tmA, &p_full[ps], g * p.cin_group_off + d.c,
                      w0 + d.dw, d.par, h0 + d.dh, n);
          if (++ps == PS) { ps = 0; pphase ^= 1; }
        }
      }
    }
  } else if (warp == 6) {
    // ------------------------------------------------ weight (B) producer --
    if (lane == 0) {
      if constexpr (WIDE) {
        mbar_expect_tx(&b_full[0], b_bytes);
        for (int i = 0; i < p.b_boxes; ++i)
          tma_load_2d(smem_b + i * p.b_box_rows * kSlabBytes, &tmB, &b_full[0], 0, i * p.b_box_rows);
      } else if constexpr (B_RESIDENT) {
        // every weight slab of the layer, once, for the life of the CTA
        const int nb = p.n_taps * p.groups;
        mbar_expect_tx(&b_full[0], nb * Cfg::kBBytes);
        for (int i = 0; i < nb; ++i) tma_load_2d(smem_b + i * Cfg::kBBytes, &tmB, &b_full[0], 0, i * BN);
      } else {
        int bs = 0;
        uint32_t bphase = 0;
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
          const int g = (tile % tiles_per_pair) / tiles_per_img;
          for (int t = 0; t < p.n_taps; ++t) {          // taps[] is already in issue order
            const int bi = g * p.n_taps + p.taps[t].b_idx;
            TWAIT(1, mbar_wait(&b_empty[bs], bphase ^ 1));
            mbar_expect_tx(&b_full[bs], Cfg::kBBytes);
            tma_load_2d(smem_b + bs * Cfg::kBBytes, &tmB, &b_full[bs], 0, bi * BN);
            if (++bs == BS) { bs = 0; bphase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // --------------------------------------------------------- MMA issuer --
    // All 32 lanes run the loops (operands stay on the uniform datapath); one elected lane issues.
    {
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint32_t a_hi = umma_desc_hi(WIDE ? 1024u : (uint32_t)p.patch_w * kSlabBytes);
      const uint32_t b_hi = umma_desc_hi(1024);
      const uint32_t p_lo0 = umma_desc_lo(smem_u32(smem_p)), p_lo_step = (uint32_t)p.patch_stage_bytes >> 4;
      const uint32_t b_lo0 = umma_desc_lo(smem_u32(smem_b));
      int ps = 0, bs = 0;
      uint32_t pphase = 0, bphase = 0;
      int it = 0;
      if constexpr (B_RESIDENT) {
        mbar_wait(&b_full[0], 0);
        tc_fence_after();
      }
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        TWAIT(4, mbar_wait(&acc_empty[acc], acc_phase ^ 1));
        tc_fence_after();
        const uint32_t d = tmem_u + acc * Cfg::kAccStride;
        int ti = 0;
        for (int pi = 0; pi < p.n_patches; ++pi) {
          const int nt = p.patches[pi].ntaps;
          TWAIT(2, mbar_wait(&p_full[ps], pphase));
          DAVO_MMA_FENCE();
          const uint32_t pa = p_lo0 + (uint32_t)ps * p_lo_step;
          for (int t = 0; t < nt; ++t, ++ti) {
            const TapDesc td = p.taps[ti];
            const uint32_t a_lo = pa + (uint32_t)td.a_off * (kSlabBytes / 16);
            uint32_t b_lo, dd = d, id = umma_idesc_tf32(kTileM, BN), acc_first = ti != 0;
            if constexpr (WIDE) {
              b_lo = b_lo0 + ((uint32_t)td.b_idx * p.b_box_rows + td.brow8 * 8u) * (kSlabBytes / 16);
              dd = d + td.dcol16 * 16u;
              id = umma_idesc_tf32(kTileM, 0) | ((uint32_t)td.n16 << 18);     // N >> 3 sits at bit 17
              acc_first = td.fresh ^ 1u;
            } else if constexpr (B_RESIDENT) {
              b_lo = b_lo0 + (uint32_t)td.b_idx * (Cfg::kBBytes / 16);        // resident: groups == 1
            } else {
              TWAIT(3, mbar_wait(&b_full[bs], bphase));
              DAVO_MMA_FENCE();
              b_lo = b_lo0 + (uint32_t)bs * (Cfg::kBBytes / 16);
            }
            if (elect_one()) tc_mma_tf32_slab(dd, a_lo, a_hi, b_lo, b_hi, id, acc_first);
            if constexpr (!B_RESIDENT) {
              if (elect_one()) tc_commit(&b_empty[bs]);   // frees the weight slot when these MMAs retire
              if (++bs == BS) { bs = 0; bphase ^= 1; }
            }
          }
          if (elect_one()) tc_commit(&p_empty[ps]);       // frees the patch slot
          if (++ps == PS) { ps = 0; pphase ^= 1; }
        }
        if (elect_one()) tc_commit(&acc_full[acc]);       // accumulator complete -> epilogue
        __syncwarp();
      }
    }
  } else {
    // ----------------------------------------------------------- epilogue --
    const int q = warp & 3;                 // TMEM lane quadrant this warp may access
    const int m = q * 32 + lane;            // accumulator row = pixel within the tile
    int it = 0;
    uint32_t epi_step = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int n = tile / tiles_per_pair;
      int r = tile - n * tiles_per_pair;
      const int g = r / tiles_per_img;
      r -= g * tiles_per_img;
      const int h = (r / p.tiles_w) * kTileH + (m >> 3);
      const int w = (r % p.tiles_w) * kTileW + (m & 7);
      const bool valid = (h < p.Hout) && (w < p.Wout);     // (unused by the WIDE store epilogue)
      const float* bias = bias_s + g * BN;
      TWAIT(5, mbar_wait(&acc_full[acc], acc_phase));
      tc_fence_after();
#ifdef DAVO_TIMING
      const long long t_busy0 = clock64();
#endif
      const uint32_t t0 = tmem_base + acc * Cfg::kAccStride + (uint32_t(q * 32) << 16);
      if constexpr (EPI == EPI_STORE_RELU && BN >= 32) {
        // 32 M rows x 32 accumulator columns per step: registers -> bias/ReLU/round -> this warp's
        // staging buffer (row = M row, 128 B, 16-B chunks XOR-swizzled by row & 7 = the tensor
        // map's 128-B swizzle) -> one TMA store of the box {32 floats, tile_w, 32/tile_w rows}.
        // TMA clips what lies outside the image.  Two buffers per warp: the store of step i
        // drains while step i+1 is computed.
        const uint32_t stg0 = smem_u32(epi_stage) + q * (FUSED ? 4096 : 8192);
        const uint32_t bias_a = smem_u32(bias_s) + g * BN * 4;
        const int c_w = (r % p.tiles_w) * TW;
        const int c_h = (r / p.tiles_w) * TH + q * (32 / TW);
#pragma unroll 1
        for (int c0 = 0; c0 < BN; c0 += 32) {
          uint32_t v[32];
          TWAIT(3, { tmem_ld_32x32(t0 + c0, v); tmem_ld_wait(); });
          const uint32_t stg = stg0 + (FUSED ? 0u : ((epi_step & 1) << 12));
          if (lane == 0) tma_store_wait_read<FUSED ? 0 : 1>();      // the store that last read this buffer is done
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 b = lds_v4(bias_a + (c0 + 4 * j) * 4);
            float4 o;
            o.x = epi_out(__uint_as_float(v[4 * j + 0]) + b.x, ea);
            o.y = epi_out(__uint_as_float(v[4 * j + 1]) + b.y, ea);
            o.z = epi_out(__uint_as_float(v[4 * j + 2]) + b.z, ea);
            o.w = epi_out(__uint_as_float(v[4 * j + 3]) + b.w, ea);
            sts_v4(stg + lane * 128 + ((j ^ (lane & 7)) << 4), o);
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_4d(&tmO, reinterpret_cast<const void*>(epi_stage + q * (FUSED ? 4096 : 8192) + (FUSED ? 0 : ((epi_step & 1) << 12))),
                         (WIDE ? 0 : g * BN) + c0, c_w, c_h, n);
            tma_store_commit();
          }
          ++epi_step;
        }
      } else if constexpr (EPI == EPI_STORE_RELU) {
        // BN = 16 (cnv1 when the widened plan does not apply): 32 pixels x 16 channels per step
        // through a swizzled staging buffer, then stores of whole 64-B runs.
        constexpr int CH = 16;
        constexpr int LPP = CH / 4;                 // lanes (float4) per pixel
        constexpr int PPS = 32 / LPP;               // pixels per store instruction
        constexpr int RB = CH * 4;                  // row bytes in the staging buffer
        uint8_t* stg = epi_stage + q * 8192;
        const int sub = lane / LPP, cq = lane % LPP;
        const int th0 = (r / p.tiles_w) * kTileH + q * 4, tw0 = (r % p.tiles_w) * kTileW;
        float* const obase = p.out + (size_t)n * p.Hout * p.Wout * p.out_stride + g * BN + cq * 4;
#pragma unroll 1
        for (int c0 = 0; c0 < BN; c0 += CH) {
          uint32_t v[CH];
          TWAIT(3, { tmem_ld_32x16(t0 + c0, v); tmem_ld_wait(); });
          __syncwarp();                             // the previous step's reads are done
#pragma unroll
          for (int j = 0; j < LPP; ++j) {
            float4 o;
            o.x = epi_out(__uint_as_float(v[4 * j + 0]) + bias[c0 + 4 * j + 0], ea);
            o.y = epi_out(__uint_as_float(v[4 * j + 1]) + bias[c0 + 4 * j + 1], ea);
            o.z = epi_out(__uint_as_float(v[4 * j + 2]) + bias[c0 + 4 * j + 2], ea);
            o.w = epi_out(__uint_as_float(v[4 * j + 3]) + bias[c0 + 4 * j + 3], ea);
            *reinterpret_cast<float4*>(stg + lane * RB + ((j ^ (lane & (LPP - 1))) << 4)) = o;
          }
          __syncwarp();
#pragma unroll
          for (int s2 = 0; s2 < 32 / PPS; ++s2) {
            const int rr = s2 * PPS + sub;          // pixel row within this warp's 32
            const float4 o = *reinterpret_cast<const float4*>(stg + rr * RB + ((cq ^ (rr & (LPP - 1))) << 4));
            const int hh = th0 + (rr >> 3), ww = tw0 + (rr & 7);
            if (hh < p.Hout && ww < p.Wout)
              *reinterpret_cast<float4*>(obase + ((size_t)hh * p.Wout + ww) * p.out_stride + c0) = o;
          }
        }
      } else {
        // Spatial-sum epilogue (cnv7 -> pred -> mean, reference nets/posenn.py:239-241:
        // pred is linear, so only sum_pixels relu(cnv7) is needed).  Each warp
        // reduces its 32 pixels per column with a transpose-reduce butterfly and
        // writes one deterministic partial row; the head kernel adds them in order.
        float* dst = p.sum_out + ((size_t)(n * p.groups + g) * tiles_per_img + r) * 4 * BN + q * BN;
        static_assert(EPI != EPI_SUM_RELU || BN >= 32, "sum epilogue wants BN >= 32");
#pragma unroll 1
        for (int c0 = 0; c0 < BN; c0 += 32) {
          uint32_t v[32];
          tmem_ld_32x32(t0 + c0, v);
          tmem_ld_wait();
          float f[32];
#pragma unroll
          for (int j = 0; j < 32; ++j)
            f[j] = valid ? fmaxf(__uint_as_float(v[j]) + bias[c0 + j], 0.f) : 0.f;
#pragma unroll
          for (int off = 16; off >= 1; off >>= 1) {
            const bool hi = (lane & off) != 0;
#pragma unroll
            for (int j = 0; j < off; ++j) {
              const float send = hi ? f[j] : f[j + off];
              const float keep = hi ? f[j + off] : f[j];
              f[j] = keep + __shfl_xor_sync(0xffffffffu, send, off);
            }
          }
          dst[c0 + lane] = f[0];            // lane L now holds column c0 + L
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[acc]);
#ifdef DAVO_TIMING
      tacc[6] += clock64() - t_busy0;
#endif
    }
    if constexpr (EPI == EPI_STORE_RELU && BN >= 32) {
      if (lane == 0) tma_store_wait_read<0>();          // shared memory must outlive the last stores
    }
  }
#ifdef DAVO_TIMING
  if (lane == 0 && (warp <= 2 || warp == 6) && blockIdx.x < 148) {
    long long* o = g_conv_timing + blockIdx.x * 8;
    if (warp == 6) o[1] = tacc[1];
    if (warp == 2) { o[7] = clock64() - t_cta0; o[0] = tacc[3]; }   // [0] reused: epilogue LDTM+wait
    if (warp == 1) { o[2] = tacc[2]; o[3] = tacc[3]; o[4] = tacc[4]; }
    if (warp == 2) { o[5] = tacc[5]; o[6] = tacc[6]; }
  }
#endif

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

}  // namespace pm
}  // namespace davo
