// Fused linear layer on tcgen05 tensor cores (sm_100a).
//
//   out[r] = residual[r] + LN( act( concat_s A_s(r) @ W + bias + gathered addends ) )
//
// One persistent 512-thread CTA per SM.  Work is cut into UNITS of 128 rows x 256 output
// columns; TMEM holds TWO 128x256 fp32 accumulators, so the epilogue of unit u overlaps
// the MMAs of unit u+1.  Two schedules:
//   N-split (n = n_valid = 512, cluster of 2): both CTAs of the cluster work on the SAME 128-row
//     tile, CTA r owning output columns [256r, 256r+256).  The A block of every K-step is
//     fetched once and multicast to both CTAs, each CTA streams only its half of the
//     weights, and LayerNorm row statistics are combined across the pair through
//     distributed shared memory.  Consecutive units of a CTA are consecutive tiles.
//   unsplit (n = 256, n_valid < 512, or a cluster of 1 or 4): every CTA walks its own tiles
//     (n/256 units per tile); the CTAs of a cluster share the weight stream by multicast.
// Warp roles:
//   warp 0        TMA lane: per K-step streams (a) 1/cluster of the pre-packed bf16 weight
//                 tile with cp.async.bulk, multicast to every CTA of the cluster, and (b)
//                 the A block of segments that are stored as operand images.
//   warp 1        MMA lane: tcgen05.mma (M=128, N=256, K=16), three products per K-step in
//                 BF16X3 mode (hi*hi, hi*lo, lo*hi), fp32 accumulation in TMEM; commits free
//                 the stage (cluster-wide) and finally publish the accumulator.
//   warp 2        TMEM allocator (512 columns).
//   warps 4-7     epilogue: tcgen05.ld (thread = row), bias, gathered pre-activation
//                 addends, swish | LayerNorm (+ residual).  fp32 outputs go through a
//                 32x32 shared-memory transpose (full 128-byte lines); operand-image
//                 outputs are written straight from the row layout (512-byte warp stores).
//                 LayerNorm needs the whole 512-wide row: statistics are accumulated over
//                 both units of a tile while the second unit's MMAs run, then both halves
//                 are normalised and their accumulators released one after the other.
//   warps 8-15    two producer groups.  A segments given as fp32 tables (optionally
//                 gathered through an index, optionally a fan-in sum) are converted to
//                 bf16 hi/lo and stored in the UMMA K-major core-matrix layout; gathered
//                 pre-activation addends (node projections of the split edge MLP) are
//                 staged into shared memory in 32-column chunks.
//
// Shared-memory operand layout (no swizzle, K-major): a [R x 16] bf16 operand of one
// K-step is two "K chunks" of 8 elements; chunk c, row r lives at byte c*LBO + r*16.
// Eight consecutive rows form one 128-byte core matrix, so SBO = 128; LBO = 256*16 for the
// weights and 128*16 + 64 for the activations (see kALbo and ptx.cuh make_smem_desc).
#pragma once
#include "../../include/graphcast_b200.h"
#include "ptx.cuh"

namespace gcb {

constexpr int kTileM = 128;
constexpr int kUnitN = 256;                       // output columns per unit / accumulator
constexpr int kKStep = 16;
constexpr int kThreads = 512;
// A operand: the two 8-element K chunks of a K-step are 2048 + 64 bytes apart.  The
// 64-byte skew puts chunk 1 on the other 16 banks so that the producers' 8-byte
// stores (rows 0-3 of both chunks per half-warp) are conflict-free.
constexpr int kALbo = kTileM * 16 + 64;           // 2112
constexpr int kAPartBytes = 2 * kALbo;            // 4224: one of {hi, lo}
constexpr int kBLbo = kUnitN * 16;                // 4096
constexpr int kBPartBytes = 2 * kBLbo;            // 8192: one of {hi, lo} of a 256-row weight block
constexpr int kEpiRowFloats = 36;                 // 32 + 4 pad: conflict-free 16 B accesses
constexpr int kEpiStageBytes = 4 * 32 * kEpiRowFloats * 4;   // per-warp 32x32 transpose tiles
// Pre-activation addend chunks (gathered node projections), double buffered:
// [2][128 rows][36 floats], filled by the producer groups, read by the epilogue.
constexpr int kGBufFloats = kTileM * kEpiRowFloats;
constexpr int kGBytes = 2 * kGBufFloats * 4;
constexpr int kMaxN = 512;
constexpr int kMaxKSteps = 128;                   // K <= 2048
constexpr int kTmemCols = 512;
static_assert(2 * kAPartBytes == GCB_A_IMAGE_BLOCK, "A image block must match the stage layout");

// Shared-memory budget: everything the variant does not need goes to pipeline stages -
// the operand ring is latency-bound (tools/pipe_rate.cu: 6 stages 411, 8 stages 389 cycles
// per K-step for a 384-cycle bf16x3 K-step).  LayerNorm variants never stage gathered
// addends (only the 2 KB statistics exchange aliases that region); the others carry no
// LayerNorm scale / offset.
constexpr int kSmemLimit = 227 * 1024;            // opt-in dynamic shared memory per CTA
constexpr int kTailBytes = 1024;                  // barriers, TMEM slot, segment tables
constexpr int kLnxBytes = 2 * kTileM * 8;         // [2][128] (mean, M2) pairs

template <bool kSplit, bool kLN>
struct TcConfig {
  static constexpr int kAStageBytes = kSplit ? 2 * kAPartBytes : kAPartBytes;
  static constexpr int kBStageBytes = kSplit ? 2 * kBPartBytes : kBPartBytes;
  static constexpr int kStageBytes = kAStageBytes + kBStageBytes;
  static constexpr int kParamBytes = (kLN ? 3 : 1) * kMaxN * 4;   // bias (, ln scale, ln offset)
  static constexpr int kGRegionBytes = kLN ? kLnxBytes : kGBytes;
  static constexpr int kFixedBytes = kParamBytes + kEpiStageBytes + kGRegionBytes + kTailBytes;
  static constexpr int kFit = (kSmemLimit - kFixedBytes) / kStageBytes;
  static constexpr int kStages = kFit < 12 ? kFit : 12;           // tail holds 2*12+10 barriers
  static constexpr int kSmemBytes = kStages * kStageBytes + kFixedBytes;
  static_assert(kStages >= 4, "operand ring too shallow");
};

__device__ __forceinline__ float swish_f(float x) {
  // x * sigmoid(x) = x / (1 + 2^(-x*log2 e)): one ex2.approx and one rcp.approx,
  // branch-free (~2 ulp), so 32 independent elements pipeline through the SFU.
  return __fdividef(x, 1.0f + __expf(-x));
}

// LayerNorm statistics of one row, fed one 32-column block (one tcgen05.ld) at a time in
// column order.  Each block's mean and M2 are taken in two passes over its registers, around
// `shift` = the mean of the row's first block, and the blocks are merged with Chan's update.
// A one-pass s2 - s1^2 / n around a single column cancels when that column lies far from
// the row mean; this stays accurate wherever an outlier sits.  The layer and the chain
// kernel both use it, so their results stay bit-identical.  The divisions are approximate
// (exact for the power-of-two counts of full blocks): an IEEE division's slow-path call
// costs the epilogue registers it does not have.
struct LnStats {
  float shift = 0.f;   // the row's values are x - shift below
  float mean = 0.f;    // mean of (x - shift) over the columns added so far
  float m2 = 0.f;      // sum of squared deviations from the mean
  float cnt = 0.f;     // columns added so far

  // x: the block's pre-LayerNorm values (overwritten); its first nv (1..32) are valid.
  __device__ __forceinline__ void add_block(float (&x)[32], int nv) {
    const float nb = static_cast<float>(nv);
    if (cnt == 0.f) {
      float p = 0.f, q = 0.f;                      // two chains for ILP
#pragma unroll
      for (int j = 0; j < 32; j += 2) {
        if (j < nv) p += x[j];
        if (j + 1 < nv) q += x[j + 1];
      }
      shift = __fdividef(p + q, nb);
    }
    float p = 0.f, q = 0.f;
#pragma unroll
    for (int j = 0; j < 32; j += 2) {
      x[j] -= shift;
      x[j + 1] -= shift;
      if (j < nv) p += x[j];
      if (j + 1 < nv) q += x[j + 1];
    }
    const float mb = __fdividef(p + q, nb);
    p = 0.f;
    q = 0.f;
#pragma unroll
    for (int j = 0; j < 32; j += 2) {
      const float d0 = x[j] - mb, d1 = x[j + 1] - mb;
      if (j < nv) p = fmaf(d0, d0, p);
      if (j + 1 < nv) q = fmaf(d1, d1, q);
    }
    const float n = cnt + nb;
    const float f = __fdividef(nb, n);
    const float d = mb - mean;
    mean = fmaf(d, f, mean);
    m2 += fmaf(d * d, cnt * f, p + q);
    cnt = n;
  }
};

// Optional timeline trace (debug): when non-null, CTA 0 records clock64() at a few
// points of each of its first kTraceTiles units; see gcb_debug_trace in api.cu.
constexpr int kTraceTiles = 64;
constexpr int kTraceEvents = 16;
__device__ long long* g_trace = nullptr;
// Debug-only experiment switches (gcb_debug_flags); 0 in production.
__device__ int g_dbg_flags = 0;

__device__ __forceinline__ void trace(uint32_t unit, int ev) {
  if (g_trace != nullptr && blockIdx.x == 0 && unit < kTraceTiles)
    g_trace[unit * kTraceEvents + ev] = clock64();
}
__device__ __forceinline__ bool tracing(uint32_t unit) {
  return g_trace != nullptr && blockIdx.x == 0 && unit < kTraceTiles;
}
__device__ __forceinline__ void trace_val(uint32_t unit, int ev, long long v) {
  if (tracing(unit)) g_trace[unit * kTraceEvents + ev] = v;
}

struct KStepInfo {
  uint8_t seg;
  uint8_t is_img;  // 1: this K-step's A block comes from the segment's operand image (TMA)
  uint16_t koff;   // element offset of this K-step inside its segment
};

// Per-segment fields copied to shared memory once: reading them from the kernel
// parameter (constant bank) inside the hot loops costs an exposed ~100-cycle LDC each.
struct SegInfo {
  const float* table;
  const int32_t* idx;
  const uint8_t* img;
  int ld, k_valid, fan, ksteps;
};
struct PreAddInfo {
  const float* table;
  const int32_t* idx;
  long long ld;
};

// kSplit: bf16x3 (hi/lo) vs single bf16 product.  kSwish / kLN: epilogue variant,
// compile-time so the per-element loops are straight-line code.
template <bool kSplit, bool kSwish, bool kLN>
__global__ void __launch_bounds__(kThreads, 1)
mlp_layer_tc_kernel(const __grid_constant__ gcb_layer_desc d) {
  using Cfg = TcConfig<kSplit, kLN>;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* stage_base = smem;
  float* s_bias = reinterpret_cast<float*>(smem + Cfg::kStages * Cfg::kStageBytes);
  float* s_scale = s_bias + kMaxN;                                  // LayerNorm variants only
  float* s_offset = s_scale + kMaxN;                                // LayerNorm variants only
  float* s_epi = s_bias + Cfg::kParamBytes / 4;                     // [4][32][36]
  float* s_g = s_epi + 4 * 32 * kEpiRowFloats;                      // [2][128][36] (not kLN)
  uint8_t* tail = reinterpret_cast<uint8_t*>(s_g) + Cfg::kGRegionBytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);          // [kStages]
  uint64_t* empty_bar = full_bar + Cfg::kStages;                   // [kStages]
  uint64_t* tmem_full_bar = empty_bar + Cfg::kStages;              // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;                    // [2]
  uint64_t* g_full_bar = tmem_empty_bar + 2;                       // [2]
  uint64_t* g_empty_bar = g_full_bar + 2;                          // [2]
  uint64_t* lnx_bar = g_empty_bar + 2;                             // [2] LayerNorm pair exchange
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(lnx_bar + 2);
  SegInfo* s_seg = reinterpret_cast<SegInfo*>(tmem_base_slot + 2);        // [3]
  PreAddInfo* s_pre = reinterpret_cast<PreAddInfo*>(s_seg + 3);           // [2]
  KStepInfo* ks_info = reinterpret_cast<KStepInfo*>(s_pre + 2);           // [kMaxKSteps]
  // [2][128] LayerNorm statistics received from the partner CTA (N-split).  Aliases the
  // addend buffers, which LayerNorm layers never use (pre_add excludes LayerNorm).
  float2* s_lnx = reinterpret_cast<float2*>(s_g);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int n = d.n;
  const int n_halves = n / kUnitN;             // units per 128-row tile (1 or 2)
  const int num_tiles = (d.rows + kTileM - 1) / kTileM;
  // Segments backed by an operand image are streamed by TMA; if every segment is,
  // the producer warps have no A work at all (a_is_img).
  int ksteps = 0;
  bool a_is_img = true;
  for (int s = 0; s < d.nseg; ++s) {
    ksteps += d.seg[s].k / kKStep;
    a_is_img = a_is_img && (d.seg[s].img != nullptr);
  }
  const int dbg = g_dbg_flags;
  uint8_t* const out_img = (dbg & 2) ? nullptr : static_cast<uint8_t*>(d.out_img);
  // Descriptor fields used inside hot loops, hoisted into registers once.
  const long long rows_total = d.rows;
  const int nseg = d.nseg;
  const int n_pre = d.n_pre_add;               // gathered pre-activation addends (0..2)
  float* const out_ptr = (dbg & 2) ? nullptr : d.out;
  float* const outy_ptr = (dbg & 2) ? nullptr : d.out_y;
  const float* const res_ptr = d.residual;
  const long long ld_out = d.ld_out, ld_outy = d.ld_out_y, ld_res = d.ld_res;
  // Cluster schedule: the CTAs of a cluster walk the K-steps of `csize` consecutive
  // tiles in lockstep and share every weight tile through TMA multicast.
  const uint32_t crank = ptx::cluster_ctarank();
  const uint32_t csize = ptx::cluster_nctarank();
  // N-split only for full 512-wide rows: its LayerNorm statistics are over all 256 columns
  // of each half, and it stores whole halves.  Any other n = 512 layer runs unsplit.
  const bool nsplit = (csize == 2) && (n_halves == 2) && (d.n_valid == n);
  const uint32_t tiles_per_iter = nsplit ? 1u : csize;       // tiles a cluster covers per iteration
  const uint32_t tile_first = ptx::cluster_id_x() * tiles_per_iter;
  const uint32_t tile_stride = ptx::num_clusters_x() * tiles_per_iter;
  const uint32_t tile_off = nsplit ? 0u : crank;             // my tile = base + tile_off
  const int units_per_tile = nsplit ? 1 : n_halves;          // units this CTA runs per tile
  const uint16_t cmask = static_cast<uint16_t>((1u << csize) - 1u);
  // (experiment, debug flag 4) N-split pair without A multicast: each CTA streams the whole
  // block itself and recycles its stages on its own MMAs only.
  const bool decouple = nsplit && (dbg & 4);

  // ---- one-time setup ---------------------------------------------------------
  for (int i = threadIdx.x; i < n; i += kThreads) {
    s_bias[i] = d.bias[i];
    if (kLN) {
      s_scale[i] = d.ln_scale[i];
      s_offset[i] = d.ln_offset[i];
    }
  }
  if (threadIdx.x == 0) {
    int ks = 0;
    for (int s = 0; s < d.nseg; ++s) {
      s_seg[s].table = d.seg[s].table;
      s_seg[s].idx = d.seg[s].idx;
      s_seg[s].img = static_cast<const uint8_t*>(d.seg[s].img);
      s_seg[s].ld = d.seg[s].ld;
      s_seg[s].k_valid = d.seg[s].k_valid;
      s_seg[s].fan = d.seg[s].fan;
      s_seg[s].ksteps = d.seg[s].k / kKStep;
    }
    for (int s = 0; s < n_pre; ++s) {
      s_pre[s].table = d.pre_add[s].table;
      s_pre[s].idx = d.pre_add[s].idx;
      s_pre[s].ld = d.pre_add[s].ld;
    }
    for (int s = 0; s < d.nseg; ++s)
      for (int k = 0; k < d.seg[s].k; k += kKStep) {
        ks_info[ks].seg = static_cast<uint8_t>(s);
        ks_info[ks].is_img = d.seg[s].img != nullptr ? 1 : 0;
        ks_info[ks].koff = static_cast<uint16_t>(k);
        ++ks;
      }
    for (int s = 0; s < Cfg::kStages; ++s) {
      // 1 TMA lane (+ 4 activation-producer warps unless A comes from images only)
      ptx::mbar_init(&full_bar[s], a_is_img ? 1 : 5);
      ptx::mbar_init(&empty_bar[s], decouple ? 1 : csize);  // tcgen05.commit of every CTA in the cluster
    }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(&tmem_full_bar[b], 1);
      ptx::mbar_init(&tmem_empty_bar[b], 4);   // 4 epilogue warps
      ptx::mbar_init(&g_full_bar[b], 4);       // 4 warps of one producer group
      ptx::mbar_init(&g_empty_bar[b], 4);      // 4 epilogue warps
      ptx::mbar_init(&lnx_bar[b], 1);          // my expect_tx; the partner's 128 st.async complete it
    }
    ptx::fence_mbar_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_base_slot, kTmemCols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::cluster_sync_all();          // barrier inits visible cluster-wide before remote arrives
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_base_slot;

  // ---- roles ------------------------------------------------------------------
  if (warp == 0) {
    // ===== TMA warp =====
    // Converged warp, every lane polls, ONE elected lane issues (see the MMA warp).  The
    // loop body is kept minimal - running pointers, ring counters, one SegInfo read per
    // segment: the issuing warp shares its scheduler with an epilogue warp, and a body of
    // ~500 cycles per K-step (table lookups + 64-bit address math + waterfall loops) made
    // this warp, not HBM or the tensor pipe, the limiter of the whole kernel.
    const uint32_t b_bytes = Cfg::kBStageBytes;                 // hi (| lo) of a 256-row block
    const size_t b_block = 2 * kBPartBytes;                     // image always holds hi|lo
    const size_t b_stride = static_cast<size_t>(n_halves) * b_block;   // next K-step, same half
    const uint32_t slice = b_bytes / csize;
    const uint32_t a_bytes = Cfg::kAStageBytes;                 // hi (| lo) block of one K-step
    const uint32_t a_half = a_bytes / 2;
    const bool b_own = (csize == 1) || nsplit;                  // my own weight block, no multicast
    const uint8_t* wimg = static_cast<const uint8_t*>(d.w_packed);
    uint32_t stage = 0, phase = 0, tu = 0;
    for (uint32_t base = tile_first; base < static_cast<uint32_t>(num_tiles); base += tile_stride) {
      const uint32_t tile = base + tile_off;
      const bool tile_ok = tile < static_cast<uint32_t>(num_tiles);   // else: dummy tile
      for (int uh = 0; uh < units_per_tile; ++uh, ++tu) {
        const int h = nsplit ? static_cast<int>(crank) : uh;          // my 256-column block
        const uint8_t* b_ptr = wimg + static_cast<size_t>(h) * b_block + (b_own ? 0u : crank * slice);
        const bool tr = tracing(tu);
        long long blocked = 0;
        for (int s = 0; s < nseg; ++s) {
          const SegInfo sg = s_seg[s];
          const bool a_copy = tile_ok && sg.img != nullptr;
          // Same tile in both CTAs of an N-split pair: each fetches half of every block and
          // multicasts it to both.
          const uint8_t* a_ptr = sg.img + static_cast<size_t>(tile) * sg.ksteps * GCB_A_IMAGE_BLOCK +
                                 (nsplit && !decouple ? crank * a_half : 0u);
          const uint32_t tx = b_bytes + (a_copy ? a_bytes : 0u);
          // (experiment, debug flag 16) L2 prefetch of the same block of my next tile
          const bool pf_next = (dbg & 16) && uh == units_per_tile - 1 &&
                               tile + tile_stride < static_cast<uint32_t>(num_tiles);
          const size_t pf_off = static_cast<size_t>(tile_stride) * sg.ksteps * GCB_A_IMAGE_BLOCK;
          for (int k = 0; k < sg.ksteps; ++k) {
            const long long w0 = tr ? clock64() : 0;
            ptx::mbar_wait(&empty_bar[stage], phase ^ 1);   // free in every CTA of the cluster
            if (tr) blocked += clock64() - w0;
            uint8_t* a_dst = stage_base + stage * Cfg::kStageBytes;
            if (ptx::elect_one()) {
              ptx::mbar_arrive_expect_tx(&full_bar[stage], tx);
              if (pf_next && a_copy) ptx::bulk_prefetch_l2(a_ptr + pf_off, nsplit ? a_half : a_bytes);
              if (a_copy) {
                if (nsplit && !decouple) ptx::bulk_g2s_multicast(a_dst + crank * a_half, a_ptr, a_half, &full_bar[stage], cmask);
                else ptx::bulk_g2s(a_dst, a_ptr, a_bytes, &full_bar[stage]);
              }
              if (b_own) {
                ptx::bulk_g2s(a_dst + Cfg::kAStageBytes, b_ptr, b_bytes, &full_bar[stage]);
              } else {
                // Same block in every CTA: each fetches 1/csize and multicasts it to all.
                ptx::bulk_g2s_multicast(a_dst + Cfg::kAStageBytes + crank * slice, b_ptr, slice,
                                        &full_bar[stage], cmask);
              }
            }
            __syncwarp();
            a_ptr += GCB_A_IMAGE_BLOCK;
            b_ptr += b_stride;
            if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
          }
        }
        if (lane == 0) trace_val(tu, 7, blocked);
      }
    }
  } else if (warp == 1) {
    // ===== MMA warp =====
    // The whole warp runs the loop on warp-uniform values and ONE elected lane issues the
    // tcgen05 instructions.  Under `if (lane == 0)` every operand is divergent and the
    // compiler wraps each UTCHMMA / UTCBAR in a vector->uniform "waterfall" loop, which
    // made the issuing thread, not the tensor pipe, the limiter (tools/pipe_rate.cu: 432 vs
    // 389 cycles per K-step).  All lanes poll: a single poller with 31 lanes parked at the
    // warp barrier is 2x slower (same benchmark, style 2).
    {
      const uint32_t idesc = ptx::make_idesc_bf16(kTileM, kUnitN);
      uint32_t stage = 0, phase = 0, u = 0;
      for (uint32_t base = tile_first; base < static_cast<uint32_t>(num_tiles); base += tile_stride) {
        for (int uh = 0; uh < units_per_tile; ++uh, ++u) {
          const uint32_t buf = u & 1;
          ptx::mbar_wait(&tmem_empty_bar[buf], ((u >> 1) & 1) ^ 1);
          ptx::tc_fence_after_sync();
          if (lane == 0) trace(u, 0);
          const uint32_t dcol = tmem_base + buf * kUnitN;
          long long starved = 0;
          const bool tr = tracing(u);
          for (int ks = 0; ks < ksteps; ++ks) {
            const long long w0 = tr ? clock64() : 0;
            ptx::mbar_wait(&full_bar[stage], phase);
            if (tr) starved += clock64() - w0;
            ptx::tc_fence_after_sync();
            if (ks == 0 && lane == 0) trace(u, 1);
            const uint32_t sa = ptx::smem_addr(stage_base + stage * Cfg::kStageBytes);
            const uint32_t sb = sa + Cfg::kAStageBytes;
            const uint64_t a_hi = ptx::make_smem_desc(sa, kALbo, 128);
            const uint64_t b_hi = ptx::make_smem_desc(sb, kBLbo, 128);
            if (ptx::elect_one()) {
              ptx::mma_bf16_ss(dcol, a_hi, b_hi, idesc, ks > 0 ? 1u : 0u);
              if (kSplit) {
                // descriptors differ only in the 16-byte-unit start address field
                const uint64_t a_lo = a_hi + (kAPartBytes >> 4);
                const uint64_t b_lo = b_hi + (kBPartBytes >> 4);
                ptx::mma_bf16_ss(dcol, a_hi, b_lo, idesc, 1u);
                ptx::mma_bf16_ss(dcol, a_lo, b_hi, idesc, 1u);
              }
              // stage reusable (cluster-wide) once these MMAs retire
              if (csize == 1 || decouple) ptx::mma_commit(&empty_bar[stage]);
              else ptx::mma_commit_multicast(&empty_bar[stage], cmask);
            }
            __syncwarp();
            if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
          }
          if (ptx::elect_one()) ptx::mma_commit(&tmem_full_bar[buf]);          // accumulator complete
          __syncwarp();
          if (lane == 0) {
            trace(u, 2);
            trace_val(u, 6, starved);
          }
        }
      }
    }
  } else if (warp >= 4 && warp < 8) {
    // ===== epilogue =====
    const int ew = warp - 4;                     // == warp % 4: TMEM lane quarter
    const uint32_t lane_base = static_cast<uint32_t>(ew * 32) << 16;
    const int n_valid = d.n_valid;
    float* my_epi = s_epi + ew * 32 * kEpiRowFloats;
    const int cg = lane & 7;                     // 16-byte column group inside the 32-col block
    const int rsub = lane >> 3;                  // row within a group of 4
    uint32_t g_count = 0;

    // LayerNorm statistics of one unit's valid columns, added to those of the earlier units.
    auto stats_unit = [&](uint32_t taddr, int col_base, int ncols, LnStats& st) {
      for (int c0 = 0; c0 < ncols; c0 += 32) {
        float v[32];
        ptx::tmem_ld32(taddr + c0, v);
        float b[32];
#pragma unroll
        for (int q = 0; q < 8; ++q)
          *reinterpret_cast<float4*>(&b[4 * q]) =
              *reinterpret_cast<const float4*>(s_bias + col_base + c0 + 4 * q);
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] += b[j];
        if (c0 + 32 <= ncols) st.add_block(v, 32);
        else st.add_block(v, ncols - c0);
      }
    };

    // Finish one unit: bias, addends, activation / normalisation, outputs.  Only one warp
    // per SM sub-partition runs this, so nothing hides latency for it: the fast path is
    // branch-free and batches its loads (residual rows are requested before the TMEM read,
    // the eight shared-memory reads are issued back to back).
    auto finish_unit = [&](uint32_t taddr, uint32_t tile, long long row0, int col_base, int ncols,
                           float mean, float rstd) {
      const bool rows_full = row0 + 32 <= rows_total;
      const bool tile_ok = tile < static_cast<uint32_t>(num_tiles);
      for (int c0 = 0; c0 < ncols; c0 += 32) {
        const int gc0 = col_base + c0;             // global column of this 32-wide block
        const int col = gc0 + cg * 4;
        const bool fast = rows_full && (c0 + 32 <= ncols);
        float4 rr[8];
        if (fast && res_ptr != nullptr) {
#pragma unroll
          for (int i = 0; i < 8; ++i)
            rr[i] = *reinterpret_cast<const float4*>(res_ptr + (row0 + rsub + 4 * i) * ld_res + col);
        }
        float v[32];
        ptx::tmem_ld32(taddr + c0, v);
        {
          float b[32];
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(&b[4 * q]) = *reinterpret_cast<const float4*>(s_bias + gc0 + 4 * q);
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] += b[j];
        }
        if (!kLN && n_pre > 0) {
          // Add the gathered node projections staged by the producer groups.
          const uint32_t gb = g_count & 1;
          ptx::mbar_wait(&g_full_bar[gb], (g_count >> 1) & 1);
          const float* gp = s_g + gb * kGBufFloats + (ew * 32 + lane) * kEpiRowFloats;
          float g[32];
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(&g[4 * q]) = *reinterpret_cast<const float4*>(gp + 4 * q);
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] += g[j];
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&g_empty_bar[gb]);
          ++g_count;
        }
        if (kSwish) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = swish_f(v[j]);
        }
        if (kLN) {
          float g[32];
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(&g[4 * q]) = *reinterpret_cast<const float4*>(s_scale + gc0 + 4 * q);
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = (v[j] - mean) * rstd * g[j];
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(&g[4 * q]) = *reinterpret_cast<const float4*>(s_offset + gc0 + 4 * q);
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] += g[j];
        }
        if (out_ptr != nullptr || outy_ptr != nullptr) {
          // 32x32 transpose through the padded per-warp tile: 8 lanes then cover one
          // 128-byte row segment and a warp store writes four complete lines.
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(my_epi + lane * kEpiRowFloats + q * 4) =
                make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
          __syncwarp();
          if (fast) {
            float4 y[8];
#pragma unroll
            for (int i = 0; i < 8; ++i)
              y[i] = *reinterpret_cast<const float4*>(my_epi + (rsub + 4 * i) * kEpiRowFloats + cg * 4);
            if (outy_ptr != nullptr) {
#pragma unroll
              for (int i = 0; i < 8; ++i)
                *reinterpret_cast<float4*>(outy_ptr + (row0 + rsub + 4 * i) * ld_outy + col) = y[i];
            }
            if (out_ptr != nullptr) {
              if (res_ptr != nullptr) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  y[i].x += rr[i].x; y[i].y += rr[i].y; y[i].z += rr[i].z; y[i].w += rr[i].w;
                }
              }
#pragma unroll
              for (int i = 0; i < 8; ++i)
                *reinterpret_cast<float4*>(out_ptr + (row0 + rsub + 4 * i) * ld_out + col) = y[i];
            }
            if (out_img != nullptr && res_ptr != nullptr) {
              // The image must hold residual + y: hand the sums back through the tile.
#pragma unroll
              for (int i = 0; i < 8; ++i)
                *reinterpret_cast<float4*>(my_epi + (rsub + 4 * i) * kEpiRowFloats + cg * 4) = y[i];
            }
          } else {
            // Ragged edge (last rows of the matrix / last partial column block).
            for (int i = 0; i < 8; ++i) {
              const int r = rsub + 4 * i;
              const long long grow = row0 + r;
              if (grow < rows_total) {
                for (int e = 0; e < 4 && c0 + cg * 4 + e < ncols; ++e) {
                  const float yv = my_epi[r * kEpiRowFloats + cg * 4 + e];
                  const float ov = yv + (res_ptr ? res_ptr[grow * ld_res + col + e] : 0.f);
                  if (outy_ptr != nullptr) outy_ptr[grow * ld_outy + col + e] = yv;
                  if (out_ptr != nullptr) out_ptr[grow * ld_out + col + e] = ov;
                  if (out_img != nullptr) my_epi[r * kEpiRowFloats + cg * 4 + e] = ov;
                }
              }
            }
          }
          __syncwarp();
          if (out_img != nullptr && res_ptr != nullptr) {
#pragma unroll
            for (int q = 0; q < 8; ++q)
              *reinterpret_cast<float4*>(&v[4 * q]) =
                  *reinterpret_cast<const float4*>(my_epi + lane * kEpiRowFloats + q * 4);
            __syncwarp();
          }
        }
        if (out_img != nullptr && tile_ok) {
          // Operand image of this tile for a later layer: thread = row, so the 16-byte
          // pieces of 32 consecutive rows are contiguous -> 512-byte coalesced warp stores.
          uint8_t* blk = out_img + (static_cast<size_t>(tile) * (n >> 4) + (gc0 >> 4)) * GCB_A_IMAGE_BLOCK +
                         (ew * 32 + lane) * 16;
#pragma unroll
          for (int ks2 = 0; ks2 < 2; ++ks2) {
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              const float* x = &v[ks2 * 16 + c * 8];
              uint2 h0, l0, h1, l1;
              ptx::split_bf16x4(make_float4(x[0], x[1], x[2], x[3]), h0, l0);
              ptx::split_bf16x4(make_float4(x[4], x[5], x[6], x[7]), h1, l1);
              uint8_t* dst = blk + ks2 * GCB_A_IMAGE_BLOCK + c * kALbo;
              *reinterpret_cast<uint4*>(dst) = make_uint4(h0.x, h0.y, h1.x, h1.y);
              *reinterpret_cast<uint4*>(dst + kAPartBytes) = make_uint4(l0.x, l0.y, l1.x, l1.y);
            }
          }
        }
      }
    };

    auto release = [&](uint32_t buf) {
      ptx::tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tmem_empty_bar[buf]);
    };

    uint32_t u = 0;
    for (uint32_t base = tile_first; base < static_cast<uint32_t>(num_tiles); base += tile_stride) {
      const uint32_t tile = base + tile_off;
      const long long row0 = static_cast<long long>(tile) * kTileM + ew * 32;
      if (!kLN) {
        for (int uh = 0; uh < units_per_tile; ++uh, ++u) {
          const int h = nsplit ? static_cast<int>(crank) : uh;
          const uint32_t buf = u & 1;
          ptx::mbar_wait(&tmem_full_bar[buf], (u >> 1) & 1);
          ptx::tc_fence_after_sync();
          if (ew == 0 && lane == 0) trace(u, 3);
          const int col_base = h * kUnitN;
          const int ncols = min(kUnitN, n_valid - col_base);
          finish_unit(tmem_base + lane_base + buf * kUnitN, tile, row0, col_base, ncols, 0.f, 1.f);
          if (ew == 0 && lane == 0) trace(u, 5);
          release(buf);
        }
      } else if (nsplit) {
        // LayerNorm over a row whose two halves live in the two CTAs of the cluster: each
        // CTA computes (mean, M2) of its 256 columns, hands them to the partner through
        // distributed shared memory, and both combine them (Chan's parallel update).
        const uint32_t buf = u & 1, par = (u >> 1) & 1;
        ptx::mbar_wait(&tmem_full_bar[buf], par);
        ptx::tc_fence_after_sync();
        if (ew == 0 && lane == 0) trace(u, 3);
        const int col_base = static_cast<int>(crank) * kUnitN;
        const uint32_t taddr = tmem_base + lane_base + buf * kUnitN;
        LnStats st;
        stats_unit(taddr, col_base, kUnitN, st);
        const float mean_h = st.shift + st.mean;                        // mean of my 256 columns
        const float m2_h = st.m2;                                       // sum of squared deviations
        const int myrow = ew * 32 + lane;
        const uint32_t peer = crank ^ 1u;
        ptx::st_async_f32x2(ptx::mapa(ptx::smem_addr(&s_lnx[buf * kTileM + myrow]), peer), mean_h, m2_h,
                            ptx::mapa(ptx::smem_addr(&lnx_bar[buf]), peer));
        if (ew == 0 && lane == 0) ptx::mbar_arrive_expect_tx(&lnx_bar[buf], kTileM * 8);
        ptx::mbar_wait(&lnx_bar[buf], par);
        const float2 other = s_lnx[buf * kTileM + myrow];
        const float delta = other.x - mean_h;
        const float mean = 0.5f * (mean_h + other.x);
        const float var = (m2_h + other.y + delta * delta * (0.5f * kUnitN)) * (1.0f / (2 * kUnitN));
        const float rstd = rsqrtf(var + 1e-5f);
        if (ew == 0 && lane == 0) trace(u, 4);
        finish_unit(taddr, tile, row0, col_base, kUnitN, mean, rstd);
        if (ew == 0 && lane == 0) trace(u, 5);
        release(buf);
        ++u;
      } else {
        // Statistics over all units of the row (overlapping the MMAs of the later ones),
        // then normalise / store unit by unit, releasing each accumulator as soon as done.
        LnStats st;
        const uint32_t u0 = u;
        for (int h = 0; h < n_halves; ++h, ++u) {
          const uint32_t buf = u & 1;
          ptx::mbar_wait(&tmem_full_bar[buf], (u >> 1) & 1);
          ptx::tc_fence_after_sync();
          if (ew == 0 && lane == 0) trace(u, 3);
          const int col_base = h * kUnitN;
          stats_unit(tmem_base + lane_base + buf * kUnitN, col_base, min(kUnitN, n_valid - col_base), st);
          if (ew == 0 && lane == 0) trace(u, 4);
        }
        const float mean = st.shift + st.mean;
        const float rstd = rsqrtf(st.m2 * (1.0f / static_cast<float>(n_valid)) + 1e-5f);
        for (int h = 0; h < n_halves; ++h) {
          const uint32_t uu = u0 + h, buf = uu & 1;
          const int col_base = h * kUnitN;
          finish_unit(tmem_base + lane_base + buf * kUnitN, tile, row0, col_base,
                      min(kUnitN, n_valid - col_base), mean, rstd);
          if (ew == 0 && lane == 0) trace(uu, 5);
          release(buf);
        }
      }
    }
  } else if (warp >= 8) {
    // ===== producers =====
    const int group = (warp - 8) >> 2;            // 0 or 1
    const int tid_g = threadIdx.x - 256 - group * 128;
    const int sub = tid_g & 3;                    // which float4 of the 16-wide K-step
    const int rg = tid_g >> 2;                    // 0..31; rows rg + 32*i
    const uint32_t sts_off = (sub >> 1) * kALbo + (sub & 1) * 8;
    const bool gather_mode = !kLN && n_pre > 0;
    // With an image-fed A operand both groups gather (alternating chunks, one buffer
    // each); otherwise group 0 produces A and group 1 gathers.
    if (gather_mode && (a_is_img || group == 1)) {
      // ----- pre-activation addend producer -----
      // Thread (rp, cgp): rows rp + 16*p (p < 8), 16-byte column group cgp of each 32-column
      // chunk: 8 lanes read one 128-byte line segment of a gathered row.
      const int cgp = tid_g & 7, rp = tid_g >> 3;
      uint32_t gc = 0;
      // Columns this CTA finishes: its own 256-wide block when N-split, else all n.
      const int gcol_lo = nsplit ? static_cast<int>(crank) * kUnitN : 0;
      const int gcol_hi = nsplit ? gcol_lo + kUnitN : n;
      for (uint32_t base = tile_first; base < static_cast<uint32_t>(num_tiles); base += tile_stride) {
        const long long trow0 = static_cast<long long>(base + tile_off) * kTileM;
        const float* p0[8];
        const float* p1[8];
#pragma unroll
        for (int p = 0; p < 8; ++p) {
          const long long grow = trow0 + rp + 16 * p;
          p0[p] = nullptr; p1[p] = nullptr;
          if (grow < rows_total) {
            const PreAddInfo a = s_pre[0];
            p0[p] = a.table + (a.idx ? static_cast<long long>(__ldg(a.idx + grow)) : grow) * a.ld + cgp * 4;
            if (n_pre > 1) {
              const PreAddInfo b = s_pre[1];
              p1[p] = b.table + (b.idx ? static_cast<long long>(__ldg(b.idx + grow)) : grow) * b.ld + cgp * 4;
            }
          }
        }
        for (int c0 = gcol_lo; c0 < gcol_hi; c0 += 32, ++gc) {
          const uint32_t gb = gc & 1;
          if (a_is_img && gb != static_cast<uint32_t>(group)) continue;
          float4 acc[8];
#pragma unroll
          for (int p = 0; p < 8; ++p)
            acc[p] = p0[p] ? __ldg(reinterpret_cast<const float4*>(p0[p] + c0)) : make_float4(0.f, 0.f, 0.f, 0.f);
          if (n_pre > 1) {
#pragma unroll
            for (int p = 0; p < 8; ++p) {
              if (p1[p]) {
                const float4 t = __ldg(reinterpret_cast<const float4*>(p1[p] + c0));
                acc[p].x += t.x; acc[p].y += t.y; acc[p].z += t.z; acc[p].w += t.w;
              }
            }
          }
          ptx::mbar_wait(&g_empty_bar[gb], ((gc >> 1) & 1) ^ 1);
          float* gdst = s_g + gb * kGBufFloats + rp * kEpiRowFloats + cgp * 4;
#pragma unroll
          for (int p = 0; p < 8; ++p)
            *reinterpret_cast<float4*>(gdst + 16 * p * kEpiRowFloats) = acc[p];
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&g_full_bar[gb]);
        }
      }
    } else if (!a_is_img) {
      // ----- activation (A operand) producer -----
      uint32_t it = 0;
      for (uint32_t base = tile_first; base < static_cast<uint32_t>(num_tiles); base += tile_stride) {
        const uint32_t tile = base + tile_off;       // may be past the end: all-zero dummy tile
        // Source row of each of my 4 tile rows, per segment (-1 = out of range).
        long long src[3][4];
#pragma unroll
        for (int s = 0; s < 3; ++s) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            src[s][i] = -1;
            if (s < nseg) {
              const long long grow = static_cast<long long>(tile) * kTileM + rg + 32 * i;
              const int32_t* ip = s_seg[s].idx;
              if (grow < rows_total) src[s][i] = ip ? static_cast<long long>(__ldg(ip + grow)) : grow;
            }
          }
        }
        for (int uh = 0; uh < units_per_tile; ++uh) {
          float4 cur[4];
          bool have_cur = false, cur_img = false;
          uint32_t cur_it = 0;
          // Software pipeline over the K-steps this group owns: the loads of the next
          // owned K-step are in flight while the current one is converted and stored.
          for (int ks = 0; ks <= ksteps; ++ks) {
            const uint32_t this_it = it + ks;
            // Normal mode: the two groups alternate K-steps.  Gather mode: group 0 owns all.
            const bool mine = (ks < ksteps) && (gather_mode || (this_it & 1u) == static_cast<uint32_t>(group));
            float4 nxt[4];
            const bool img_step = mine && ks_info[ks].is_img;   // TMA brings the data: arrive only
            if (mine && !img_step) {
              const int s = ks_info[ks].seg;
              const int koff = ks_info[ks].koff + sub * 4;
              const SegInfo sg = s_seg[s];
              const bool kvalid = koff < sg.k_valid;
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                const long long sr = (s == 0) ? src[0][i] : (s == 1 ? src[1][i] : src[2][i]);
                if (kvalid && sr >= 0) {
                  const float* p = sg.table + sr * sg.fan * sg.ld + koff;
                  acc = __ldg(reinterpret_cast<const float4*>(p));
                  for (int j = 1; j < sg.fan; ++j) {
                    const float4 t = __ldg(reinterpret_cast<const float4*>(p + static_cast<long long>(j) * sg.ld));
                    acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w;
                  }
                }
                nxt[i] = acc;
              }
            }
            if (have_cur && (mine || ks == ksteps)) {
              const uint32_t stage = cur_it % Cfg::kStages;
              const uint32_t phase = (cur_it / Cfg::kStages) & 1;
              ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
              uint8_t* a_hi = stage_base + stage * Cfg::kStageBytes;
              if (!cur_img) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                  uint2 hi, lo;
                  ptx::split_bf16x4(cur[i], hi, lo);
                  const uint32_t off = sts_off + (rg + 32 * i) * 16;
                  *reinterpret_cast<uint2*>(a_hi + off) = hi;
                  if (kSplit) *reinterpret_cast<uint2*>(a_hi + kAPartBytes + off) = lo;
                }
              }
              ptx::fence_proxy_async_smem();
              __syncwarp();
              if (lane == 0) ptx::mbar_arrive(&full_bar[stage]);
              have_cur = false;
            }
            if (mine) {
#pragma unroll
              for (int i = 0; i < 4; ++i) cur[i] = nxt[i];
              cur_it = this_it;
              cur_img = img_step;
              have_cur = true;
            }
          }
          it += ksteps;
        }
      }
    }
  }

  // ---- teardown ---------------------------------------------------------------
  // No CTA may exit while a peer can still multicast into its shared memory or arrive
  // on its barriers.
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::cluster_sync_all();
  if (warp == 2) {
    ptx::tc_fence_after_sync();
    ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

}  // namespace gcb
